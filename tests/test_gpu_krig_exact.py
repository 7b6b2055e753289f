"""ked_kernel (twxi_krig) against a 40-digit restatement of gstat's kriging with external drift.

The float64 oracle is 1e-4 C away from the kernel's own accuracy in test_gpu_parity, which a kernel that lost six digits
would pass.  The referee here is ``ked_exact``: the uncentred augmented system of universal kriging
    [[V, F], [F', 0]] [lambda; mu] = [c0; f0],   F = [1, lon, lat, elev, lst_m],   f0 = F of the point,
    mean = lambda'y,   var = C(0) - lambda'c0 - mu'f0,
built and solved to 1e-35 in 40-digit arithmetic from the kernel's own float64 inputs (neighbours, counts, variogram,
station table).  Each tolerance is a first-order componentwise bound from the problem itself (``_bounds``), with one
documented multiplier C_BOUND.  Measured on a B200 (1 000 W power limit), the kernel's worst error / bound is 0.036 for
the mean and 0.26 for the variance, and each of these changes to it fails this file: dropping the c5 term of the
covariance polynomial (at most 3.9e-14 relative, odd in f, so its sign varies from pair to pair: test E's predictions
next to a station, whose variance hangs on one covariance at f = -0.499, reach 1.7-2.2; every other case stays below
0.7), a second-order pivot reciprocal (up to 9x), four pivots instead of five in the 5x5 trend solve (1e12x), and
accepting fewer than 5 neighbours (test F).

Covered: every size class NB = ceil(n/8) = 1..21 at n = 8 NB - 7 and 8 NB (168 = TWXI_MAX_KRIG_NNGHS), n = 5, 6, 7, all
classes in one shuffled call, each point also bitwise equal to itself solved alone; the production path (smoothed counts
and variogram, mth = 0 against every single month); every launch variant; CTAs that solve many problems in a row, with
failing points interleaved, bitwise equal to one point per staging sub-batch; the pure nugget model (range 0, psill 0),
nugget 0, the -250/km clamp of the range, underflowing covariances, prediction at a station; fewer than 5 neighbours.

Known gap (out of scope): a drift that is rank deficient with n >= 5 (say every neighbour with one LST value) is
singular in exact arithmetic, but no exact test of it exists without a threshold; such points are decided by the rounded
pivots.

Run with -m gpu; the reference's own checks run on the CPU."""
import multiprocessing as mp
import os

import numpy as np
import pytest

mpmath = pytest.importorskip("mpmath")      # comes with torch (through sympy)
sla = pytest.importorskip("scipy.linalg")

from oracle import twx_oracle as o          # noqa: E402

DPS = 40
EPS = 2.0 ** -53
C_BOUND = 64                                # bound = C_BOUND * eps * (first-order terms), as in test_gpu_gwr_exact
# Relative error allowed for the device's gcdist_sp, in units of eps.  With the degree -> radian products taken as
# gcdist_sp forms them (see gcdist_exact), numpy's float64 gcdist_sp measures <= 5.6 eps against gcdist_exact here
# (test_host_distance_error_fits_c_h keeps it <= C_H / 4).  CUDA documents sin, cos, sincos and atan to 2 ulp, glibc
# to < 1 ulp: the device may have twice the host's error, and a factor 2 is left on top.  The device's own distance
# error cannot be observed through the C ABI (twxi_knn returns the haversine distances, not these).
C_H = 32
REFINE_TOL = 1e-35
REFINE_STEPS = 6
GUARD = 10                                  # guard digits of the residuals: K is uncentred (elevations in metres), so a
                                            # DPS-digit residual alone stalls the refinement near 1e-34 at cond(K) ~ 1e6
MAX_N = 168                                 # TWXI_MAX_KRIG_NNGHS
ST_OK, ST_SINGULAR, ST_LIMIT = 0, 4, 8
DE2RA = np.pi / 180.0                       # the float64 constant of gcdist_sp
COUNTS_A = sorted({5, 6, 7, 8} | {8 * nb - 7 for nb in range(2, 22)} | {8 * nb for nb in range(2, 22)})
VARIOS = {"typical": (0.2, 1.1, 120.0), "short range": (0.3, 1.0, 12.0), "long range": (1e-3, 1.5, 900.0)}
MTH_A = 5


# ---- the reference --------------------------------------------------------------------------------------------------
def _mp(x):
    return mpmath.mpf(float(x))


def gcdist_exact(lon1, lat1, lon2, lat2):
    """gcdist_sp (Andoyer-Lambert, WGS-84) at DPS digits, with its exact-zero rule for co-located points.  The degree ->
    radian products are the float64 ones gcdist_sp forms: from there the latitude and longitude differences are exact in
    float64 (Sterbenz), and everything after them is evaluated exactly.  Rounded at 1e-16 rad, those products would
    otherwise move a 1 km distance by 1e-12 relative in any float64 implementation, and say nothing about the kernel."""
    eps = 2.220446049250313e-16
    if abs(lat1 - lat2) < eps and (abs(lon1 - lon2) < eps or abs((abs(lon1) + abs(lon2)) - 360.0) < eps):
        return mpmath.mpf(0)
    fl = 1 / mpmath.mpf("298.257223563")
    a, b = _mp(lat1 * DE2RA), _mp(lat2 * DE2RA)
    c, d = _mp(lon1 * DE2RA), _mp(lon2 * DE2RA)
    F, G, L = (a + b) / 2, (a - b) / 2, (c - d) / 2
    sG, cG, sF, cF = mpmath.sin(G), mpmath.cos(G), mpmath.sin(F), mpmath.cos(F)
    sL, cL = mpmath.sin(L), mpmath.cos(L)
    S = sG ** 2 * cL ** 2 + cF ** 2 * sL ** 2
    C = cG ** 2 * cL ** 2 + sF ** 2 * sL ** 2
    w = mpmath.atan(mpmath.sqrt(S / C))
    R = mpmath.sqrt(S * C) / w
    H1, H2 = (3 * R - 1) / (2 * C), (3 * R + 1) / (2 * S)
    return 2 * w * mpmath.mpf("6378.137") * (1 + fl * H1 * sF ** 2 * cG ** 2 - fl * H2 * cF ** 2 * sG ** 2)


def cov_exact(h, vario):
    """gstat's covariance (oracle.covariance_gstat) at DPS digits: nug + psill at h == 0, psill exp(-h / range) beyond,
    0 beyond for the pure nugget model (range == 0)."""
    nug, psill, rng = (_mp(v) for v in vario)
    if h == 0:
        return nug + psill
    if rng == 0:
        return mpmath.mpf(0)
    return psill * mpmath.exp(-h / rng)


def _bounds(V, c0, Fc, y, D, d0, c00):
    """First-order componentwise bounds of |mean error|, |var error| in the kernel's parametrisation (drift centred on
    the point and scaled by (1, 1, 1, 1e-3, 0.1), y - yref with yref the first neighbour's value), float64:
        s = Kc^-1 rc, w = Kc^-1 [y - yref; 0],  Kc = [[V, Fc], [Fc', 0]],  rc = [c0; e0];
        |dmean| <= C u (|w|'(|Kc||s| + |rc|) + |lambda|'|y - yref| + |yref|) + C_H u |w|'(D|s| + d0)
        |dvar|  <= C u (C(0) + 2|s|'|rc| + |s|'|Kc||s|) + C_H u (2|s|'d0 + |s|'D|s|)
    D_ij = C(h_ij) h_ij / range and d0_j = C(h_0j) h_0j / range: the first-order change of the covariances under a
    relative distance error.
    The kernel forms S = A'A, A = L^-1 [Fc, y - yref, c0] (V = LL'), explicitly and then eliminates its trend block
    (ked.cu).  The backward error of that elimination is |K| in the V and Fc blocks but |A|'|A| in the zero trend block
    of K, so both bounds get the first-order effect of |dS| <= C u |A|'|A| on top:
        |dmean| += C u (|A||p|)'(|A||q|),   |dvar| += C u (|A||q|)'(|A||q|),
    p = [-G^-1 g_y; 1; 0], q = [G^-1 (e0 - g_c); 0; 1] (mean - yref = p'S q and var = C(0) - q'S q to first order).
    This term dominates only where the explicit S does lose digits: few neighbours, short ranges."""
    n = y.size
    N = n + 5
    Kc = np.zeros((N, N))
    Kc[:n, :n], Kc[:n, n:], Kc[n:, :n] = V, Fc, Fc.T
    rc = np.concatenate([c0, [1.0, 0, 0, 0, 0]])
    yc = np.concatenate([y - y[0], np.zeros(5)])
    lu = sla.lu_factor(Kc)
    s, w = np.abs(sla.lu_solve(lu, rc)), np.abs(sla.lu_solve(lu, yc))
    A = np.abs(Kc)
    Df = np.zeros((N, N))
    Df[:n, :n] = D
    df = np.concatenate([d0, np.zeros(5)])
    u = EPS
    mb = (C_BOUND * u * (w @ (A @ s + np.abs(rc)) + s[:n] @ np.abs(yc[:n]) + abs(y[0]))
          + C_H * u * (w @ (Df @ s + df)))
    vb = C_BOUND * u * (c00 + 2 * s @ np.abs(rc) + s @ A @ s) + C_H * u * (2 * s @ df + s @ Df @ s)
    Ab = sla.solve_triangular(np.linalg.cholesky(V), np.column_stack([Fc, yc[:n], c0]), lower=True)
    S = Ab.T @ Ab
    p = np.concatenate([-np.linalg.solve(S[:5, :5], S[:5, 5]), [1.0, 0.0]])
    q = np.concatenate([np.linalg.solve(S[:5, :5], np.eye(5)[0] - S[:5, 6]), [0.0, 1.0]])
    ap, aq = np.abs(Ab) @ np.abs(p), np.abs(Ab) @ np.abs(q)
    mb += C_BOUND * u * (ap @ aq)
    vb += C_BOUND * u * (aq @ aq)
    return float(mb), float(vb)


def ked_exact(X, y, x0, vario, H, h0, keep=False):
    """Kriging with external drift of one problem at DPS digits.

    X [n][4] station (lon, lat, elev, lst_m) and y [n] normals (float64, taken as exact), x0 the point's (lon, lat,
    elev, lst_m), vario (nug, psill, range), H [n][n] and h0 [n] the exact distances (gcdist_exact).  The indefinite K is
    solved by float64 LU of its centred and scaled form (a preconditioner only) and iterative refinement with residuals
    at DPS + GUARD digits until the correction is below REFINE_TOL relative; mpmath.lu_solve if REFINE_STEPS do not get
    there.
    Returns dict(mean, var (mpf), mean_bound, var_bound, steps, converged[, lam, mu, F, f0])."""
    with mpmath.workdps(DPS):
        n = len(y)
        N = n + 5
        h0 = h0[:n]                         # H and h0 may be those of a longer neighbour list (leading blocks)
        X = np.asarray(X, dtype=np.float64)
        y = np.asarray(y, dtype=np.float64)
        x0 = np.asarray(x0, dtype=np.float64)
        c00 = _mp(vario[0]) + _mp(vario[1])
        K = np.empty((N, N), dtype=object)
        K[n:, n:] = mpmath.mpf(0)
        for i in range(n):
            K[i, i] = c00
            for j in range(i):
                K[i, j] = K[j, i] = cov_exact(H[i][j], vario)
        F = np.empty((n, 5), dtype=object)
        F[:, 0] = mpmath.mpf(1)
        for a in range(4):
            F[:, a + 1] = [_mp(v) for v in X[:, a]]
        K[:n, n:], K[n:, :n] = F, F.T
        c0 = np.array([cov_exact(h, vario) for h in h0], dtype=object)
        f0 = np.array([mpmath.mpf(1)] + [_mp(v) for v in x0], dtype=object)
        r = np.concatenate([c0, f0])
        # preconditioner: the centred, scaled system Kc = P' K P, P = diag(I, T), F T = Fc
        sc = np.array([1.0, 1.0, 1e-3, 0.1])
        Fc = np.column_stack([np.ones(n), (X - x0) * sc])
        T = np.diag(np.concatenate([[1.0], sc]))
        T[0, 1:] = -x0 * sc
        V64 = np.array([[float(v) for v in row] for row in K[:n, :n]])
        Kc = np.zeros((N, N))
        Kc[:n, :n], Kc[:n, n:], Kc[n:, :n] = V64, Fc, Fc.T
        lu = sla.lu_factor(Kc)

        def inv(v):
            v = np.array(v, dtype=np.float64)
            v[n:] = T.T @ v[n:]
            z = sla.lu_solve(lu, v)
            z[n:] = T @ z[n:]
            return z
        x = np.array([_mp(v) for v in inv([float(v) for v in r])], dtype=object)
        steps, converged = 0, False
        while steps < REFINE_STEPS:
            steps += 1
            with mpmath.workdps(DPS + GUARD):
                d = inv([float(v) for v in r - K.dot(x)])
                x = x + d
            if np.abs(d).max() <= REFINE_TOL * max(abs(float(v)) for v in x):
                converged = True
                break
        if not converged:
            sol = mpmath.lu_solve(mpmath.matrix(K.tolist()), mpmath.matrix(r.tolist()))
            x = np.array([sol[i] for i in range(N)], dtype=object)
        lam, mu = x[:n], x[n:]
        mean = mpmath.fdot(lam, [_mp(v) for v in y])
        var = c00 - mpmath.fdot(lam, c0) - mpmath.fdot(mu, f0)
        # bounds, float64
        rng = float(vario[2])
        smooth = rng > 0 and float(vario[1]) != 0
        Hf = np.array([[float(H[i][j]) for j in range(n)] for i in range(n)])
        h0f = np.array([float(h) for h in h0])
        D = np.abs(V64) * Hf / rng if smooth else np.zeros((n, n))
        c0f = np.array([float(v) for v in c0])
        d0 = np.abs(c0f) * h0f / rng if smooth else np.zeros(n)
        mb, vb = _bounds(V64, c0f, Fc, y, D, d0, float(c00))
        out = dict(mean=mean, var=var, mean_bound=mb, var_bound=vb, steps=steps, converged=converged)
        if keep:
            out.update(lam=lam, mu=mu, F=F, f0=f0)
        return out


def _pair_task(chunk):
    with mpmath.workdps(DPS):
        return [gcdist_exact(*p) for p in chunk]


_SHARED = {}                                # per-problem inputs, inherited by the forked workers of reference()


def _problem_task(i):
    X, y, x0, vario, gid, keep = _SHARED["probs"][i]
    H, h0 = _SHARED["dist"][gid]
    return ked_exact(X, y, x0, vario, H, h0, keep)


def _pool_map(fn, tasks):
    n = max(1, os.cpu_count() or 1)
    with mp.get_context("fork").Pool(n) as pool:
        return pool.map(fn, tasks, chunksize=1)


def reference(stns, problems, keep=False):
    """ked_exact of every problem, farmed over the host cores.  A problem is dict(gid, pt (lon, lat, elev, lst_m), sids
    (context station indices in the kernel's neighbour order), mth, vario); the problems of one gid share pt[:2] and
    the neighbour order.  Returns the results in the order of ``problems``."""
    from topowx_b200 import db
    lon, lat = np.asarray(stns[db.LON], dtype=np.float64), np.asarray(stns[db.LAT], dtype=np.float64)
    groups = {}
    for i, p in enumerate(problems):
        groups.setdefault(p["gid"], []).append(i)
    pairs, keys = [], {}
    for gid, members in groups.items():
        sids = max((problems[i]["sids"] for i in members), key=len)
        plon, plat = problems[members[0]]["pt"][:2]
        for a, s in enumerate(sids):
            for key, pt in [(("p", plon, plat, int(s)), (plon, plat, lon[s], lat[s]))] + \
                           [((int(min(s, t)), int(max(s, t))), (lon[s], lat[s], lon[t], lat[t])) for t in sids[:a]]:
                if key not in keys:
                    keys[key] = len(pairs)
                    pairs.append(pt)
    nc = 8 * max(1, os.cpu_count() or 1)
    chunks = [pairs[i::nc] for i in range(nc)]
    got = _pool_map(_pair_task, chunks)
    dist = [None] * len(pairs)
    for c, vals in enumerate(got):
        dist[c::nc] = vals
    # the distances of a group (the longest neighbour list of its point) are shared by its problems; the problems go to
    # the pool one by one, largest first, so that every core works
    _SHARED["dist"], _SHARED["probs"] = {}, [None] * len(problems)
    for gid, members in groups.items():
        sids = max((problems[i]["sids"] for i in members), key=len)
        plon, plat = problems[members[0]]["pt"][:2]
        H = [[dist[keys[(int(min(s, t)), int(max(s, t)))]] if s != t else mpmath.mpf(0) for t in sids] for s in sids]
        _SHARED["dist"][gid] = (H, [dist[keys[("p", plon, plat, int(s))]] for s in sids])
        for i in members:
            p = problems[i]
            s = p["sids"]
            assert np.array_equal(s, sids[:len(s)])
            m = p["mth"]
            X = np.column_stack([lon[s], lat[s], stns[db.ELEV][s], stns[db.get_lst_varname(m)][s]])
            _SHARED["probs"][i] = (X, np.asarray(stns[db.get_norm_varname(m)][s], dtype=np.float64), p["pt"],
                                   p["vario"], gid, keep)
    order = sorted(range(len(problems)), key=lambda i: -len(problems[i]["sids"]))
    try:
        out = _pool_map(_problem_task, order)
    finally:
        _SHARED.clear()
    res = [None] * len(problems)
    for i, r in zip(order, out):
        res[i] = r
    return res, dict(pairs=pairs, dist=dist)


class _Stats(object):
    """Worst error / bound ratio per key."""

    def __init__(self):
        self.d = {}

    def add(self, key, ratio):
        self.d[key] = max(self.d.get(key, 0.0), float(ratio))

    def report(self, title):
        print("\n" + title)
        for key in sorted(self.d):
            print("  %-48s worst error/bound %.3g" % (key, self.d[key]))


def _check(stats, key, ref, mean, var, bad, what):
    """Kernel mean / var against ked_exact within the bounds; ratios into stats."""
    em = abs(float(ref["mean"] - _mp(mean)))
    ev = abs(float(ref["var"] - _mp(var)))
    stats.add(key + " mean", em / ref["mean_bound"])
    stats.add(key + " var", ev / ref["var_bound"])
    if not (ref["converged"] and em <= ref["mean_bound"] and ev <= ref["var_bound"]):
        bad.append((what, ref["converged"], em, ref["mean_bound"], ev, ref["var_bound"]))


# ---- fixtures -------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def env():
    from topowx_b200 import synth, db
    f = synth.Fields()
    days = synth.make_days(1995, 1)
    da = synth.make_station_db(0, 2000, synth.tile_bbox(), f, days)
    mask = np.isnan(da.stns[db.BAD])
    stns = da.stns[mask]
    ss = o.StationSelect(o.StationDb(da.stns, da.var, da.days), mask)

    def nbrs(lat, lon, k):
        ss._set_pt(lat, lon)
        return ss.pt_sort_idx[:k].copy()
    return dict(f=f, days=days, da=da, mask=mask, stns=stns, nbrs=nbrs, synth=synth, db=db)


def _cells(env, rows, cols, w=0):
    synth, f = env["synth"], env["f"]
    lat, lon = synth.grid_lats(np.asarray(rows) + synth.TILE_ROW0), synth.grid_lons(np.asarray(cols) + synth.TILE_COL0)
    elev = f.elev(lon, lat)
    lst = np.stack([f.lst(w, m, lon, lat, elev) for m in range(1, 13)], axis=1)
    return lat, lon, elev, lst


@pytest.fixture(scope="module")
def case_a(env):
    """Three tile cells x every count of COUNTS_A x the three variogram sets, month MTH_A: problems in batch order."""
    lat, lon, elev, lst = _cells(env, [37, 121, 208], [190, 64, 133])
    pts = [(q, n, v) for q in range(3) for n in COUNTS_A for v in VARIOS]
    probs = []
    for q, n, v in pts:
        sids = env["nbrs"](lat[q], lon[q], MAX_N)
        probs.append(dict(gid=(q, v), pt=(lon[q], lat[q], elev[q], lst[q, MTH_A - 1]), sids=sids[:n], mth=MTH_A,
                          vario=VARIOS[v]))
    ref, dist = reference(env["stns"], probs)
    return dict(lat=lat, lon=lon, elev=elev, lst=lst, pts=pts, ref=ref, dist=dist)


E_VARIOS = {"pure nugget, range 0": (0.4, 0.9, 0.0), "pure nugget, psill 0": (1.3, 0.0, 80.0),
            "nugget 0": (0.0, 1.2, 60.0), "range 3 m (-250/km clamp)": (0.2, 1.0, 0.003),
            "range 50 m (exp below 2^-1000)": (0.2, 1.0, 0.05)}
E_COUNTS = (12, 60)


@pytest.fixture(scope="module")
def case_e(env):
    """Covariance domain: two tile cells x E_COUNTS x E_VARIOS, predictions at two stations (no rm_zero), and four
    predictions next to a station whose variance carries one covariance at the worst point of its polynomial."""
    from topowx_b200 import db
    lat, lon, elev, lst = _cells(env, [88, 170], [22, 231])
    s = env["stns"]
    on = env["nbrs"](float(lat[0]), float(lon[0]), 40)[[3, 31]]     # two stations near the first cell
    lat = np.concatenate([lat, s[db.LAT][on]])
    lon = np.concatenate([lon, s[db.LON][on]])
    elev = np.concatenate([elev, s[db.ELEV][on]])
    lst = np.concatenate([lst, np.stack([s[db.get_lst_varname(m)][on] for m in range(1, 13)], axis=1)])
    pts = [(q, n, v) for q in range(2) for n in E_COUNTS for v in E_VARIOS]
    pts += [(q, n, v) for q in (2, 3) for n in (5, 30) for v in ("typical", "nugget 0")]
    varios = dict(E_VARIOS, typical=VARIOS["typical"])
    # next to a station: four tile cells 0.15-0.6 km from their nearest station, nugget 0 and the range that puts that
    # pair at f = -0.499 of the covariance polynomial (ncov_pos: u = -h T / (range ln2), f = u - rint(u)), where its
    # highest terms weigh most.  The variance then hangs on that one covariance: -2 lambda_1 dc0_1 with lambda_1 ~ 1.
    rng = np.random.default_rng(1021)
    near = []
    while len(near) < 4:
        r, cc = rng.integers(0, 250, 2)
        la, lo, el, ls = _cells(env, [r], [cc])
        j = env["nbrs"](la[0], lo[0], 1)[0]
        h = float(o.gcdist_sp(lo[0], la[0], s[db.LON][j], s[db.LAT][j]))
        if 0.15 <= h <= 0.6:
            near.append((la, lo, el, ls))
            varios["next to a station %d" % len(near)] = (0.0, 1.0, h * 64 / (0.499 * np.log(2)))
    for k, (la, lo, el, ls) in enumerate(near):
        lat, lon, elev, lst = (np.concatenate([a, b]) for a, b in zip((lat, lon, elev, lst), (la, lo, el, ls)))
        pts.append((4 + k, 20, "next to a station %d" % (k + 1)))
    probs = []
    for q, n, v in pts:
        sids = env["nbrs"](lat[q], lon[q], n)
        probs.append(dict(gid=(q, n, v), pt=(lon[q], lat[q], elev[q], lst[q, MTH_A - 1]), sids=sids, mth=MTH_A,
                          vario=varios[v]))
    ref, dist = reference(env["stns"], probs)
    return dict(lat=lat, lon=lon, elev=elev, lst=lst, pts=pts, ref=ref, dist=dist, varios=varios, on=on)


F_ROWS, F_COLS = [3, 40, 77, 101, 150, 199, 230, 12], [9, 222, 57, 140, 18, 96, 175, 245]


@pytest.fixture(scope="module")
def case_f(env):
    """n = 5 and 6 at eight tile cells (n = 1..4 there have no reference: TWXI_ST_SINGULAR)."""
    lat, lon, elev, lst = _cells(env, F_ROWS, F_COLS)
    probs = [dict(gid=(q, n), pt=(lon[q], lat[q], elev[q], lst[q, MTH_A - 1]), sids=env["nbrs"](lat[q], lon[q], n),
                  mth=MTH_A, vario=VARIOS["typical"]) for q in range(lat.size) for n in (5, 6)]
    ref, _ = reference(env["stns"], probs)
    return dict(lat=lat, lon=lon, elev=elev, lst=lst, ref=ref)


def _ctx(env, da=None):
    from topowx_b200.context import TwxiContext
    da = env["da"] if da is None else da
    return TwxiContext(da, np.isnan(da.stns[env["db"].BAD]))


def _assert_knn(ctx, env, lat, lon, k):
    idx, _, _, st = ctx.knn(lat, lon, k)                             # k + 1 candidates per point
    assert np.all(st == 0)
    for q in range(np.size(lat)):
        assert np.array_equal(idx[q, :k], env["nbrs"](lat[q], lon[q], k)), q
    return idx[:, :k]


def _batch_a(case):
    """Case A as one shuffled batch: arrays in batch order and the permutation (batch row -> problem)."""
    perm = np.random.default_rng(20261021).permutation(len(case["pts"]))
    q = np.array([case["pts"][i][0] for i in perm])
    nn = np.array([case["pts"][i][1] for i in perm], dtype=np.int32)
    vo = np.array([VARIOS[case["pts"][i][2]] for i in perm])
    return perm, (case["lat"][q], case["lon"][q], case["elev"][q], case["lst"][q]), nn, vo


# ---- A. every size class --------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_every_size_class_vs_exact(env, case_a):
    """n = 5..8 and 8 NB - 7, 8 NB for NB = 2..21, three variogram sets, all in one shuffled call: within the bounds,
    and each point bitwise equal to itself solved alone."""
    ctx = _ctx(env)
    _assert_knn(ctx, env, case_a["lat"], case_a["lon"], MAX_N)
    perm, (lat, lon, elev, lst), nn, vo = _batch_a(case_a)
    assert {(n + 7) // 8 for n in nn} == set(range(1, 22))
    mean, var, st = ctx.krig(lat, lon, elev, lst, mth=MTH_A, nnghs=nn, vario=vo)
    assert np.all(st == ST_OK)
    stats, bad = _Stats(), []
    for b, i in enumerate(perm):
        q, n, v = case_a["pts"][i]
        _check(stats, "NB %2d %s" % ((n + 7) // 8, v), case_a["ref"][i], mean[b, 0], var[b, 0], bad, (q, n, v))
        m1, v1, s1 = ctx.krig(lat[b], lon[b], elev[b], lst[b], mth=MTH_A, nnghs=nn[b], vario=vo[b])
        assert s1[0] == ST_OK
        if not (m1[0, 0] == mean[b, 0] and v1[0, 0] == var[b, 0]):
            bad.append(("alone != batch", q, n, v))
    stats.report("A. kriging kernel against ked_exact, every size class")
    assert not bad, (len(bad), bad[:10])


# ---- B. production path ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_production_path_vs_exact(env):
    """mth = 0 with the smoothed counts and variogram of nngh_params on 24 tile cells (four clusters of six): a point's
    months fall into different size classes and read leading blocks of one staged block.  Within the bounds, and bitwise
    equal to each single-month call."""
    rows = np.concatenate([r + np.array([0, 0, 0, 1, 1, 1]) for r in (14, 92, 160, 231)])
    cols = np.concatenate([c + np.array([0, 1, 2, 0, 1, 2]) for c in (200, 35, 118, 70)])
    lat, lon, elev, lst = _cells(env, rows, cols)
    ctx = _ctx(env)
    kn, _, vario, st0 = ctx.nngh_params(lat, lon)
    assert np.all(st0 == ST_OK)
    assert len({(k + 7) // 8 for k in kn.ravel()}) >= 4
    mean, var, st = ctx.krig(lat, lon, elev, lst, mth=0)
    assert np.all(st == ST_OK)
    for m in range(1, 13):
        m1, v1, s1 = ctx.krig(lat, lon, elev, lst, mth=m)
        assert np.all(s1 == ST_OK)
        assert np.array_equal(m1[:, 0], mean[:, m - 1]) and np.array_equal(v1[:, 0], var[:, m - 1]), m
    idx = _assert_knn(ctx, env, lat, lon, int(kn.max()))
    probs, at = [], []
    for q in range(lat.size):
        for m in range(1, 13):
            probs.append(dict(gid=q, pt=(lon[q], lat[q], elev[q], lst[q, m - 1]), sids=idx[q, :kn[q, m - 1]], mth=m,
                              vario=tuple(vario[q, m - 1])))
            at.append((q, m))
    ref, _ = reference(env["stns"], probs)
    stats, bad = _Stats(), []
    for (q, m), r in zip(at, ref):
        _check(stats, "production", r, mean[q, m - 1], var[q, m - 1], bad, (q, m, kn[q, m - 1]))
    stats.report("B. production path against ked_exact")
    assert not bad, (len(bad), bad[:10])


# ---- C. launch variants ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_every_launch_variant_vs_exact(env, case_a):
    """Batch A on a fresh context per launch variant (TWXI_KED_VAR = that variant's index for every size class; the
    library moves a class to a wider variant where the chosen one is too small): within the bounds, and bitwise equal
    to the default variant table."""
    import re
    src = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "topowx_b200", "csrc",
                            "ked.cu")).read()
    nvar = len(re.findall(r"\{ked_kernel<\d+, \d+, \d+>", src))
    assert nvar == 6
    perm, (lat, lon, elev, lst), nn, vo = _batch_a(case_a)
    base = _ctx(env).krig(lat, lon, elev, lst, mth=MTH_A, nnghs=nn, vario=vo)
    stats, bad, same = _Stats(), [], []
    old = os.environ.get("TWXI_KED_VAR")
    try:
        for v in range(nvar):
            os.environ["TWXI_KED_VAR"] = str(v) * 21
            mean, var, st = _ctx(env).krig(lat, lon, elev, lst, mth=MTH_A, nnghs=nn, vario=vo)
            assert np.all(st == ST_OK), v
            for b, i in enumerate(perm):
                q, n, vn = case_a["pts"][i]
                _check(stats, "variant %d" % v, case_a["ref"][i], mean[b, 0], var[b, 0], bad, (v, q, n, vn))
            same.append(np.array_equal(mean, base[0]) and np.array_equal(var, base[1]))
    finally:
        if old is None:
            os.environ.pop("TWXI_KED_VAR", None)
        else:
            os.environ["TWXI_KED_VAR"] = old
    stats.report("C. launch variants against ked_exact")
    print("  bitwise equal to the default variant table: %s" % same)
    assert not bad, (len(bad), bad[:10])
    # every variant accumulates each tile in the same order (stage_rows: the J loop, two chains, is the same for any
    # number of workers), so the variants agree to the bit
    assert all(same), same


# ---- D. multi-problem CTAs and sub-batches --------------------------------------------------------------------------
@pytest.mark.gpu
def test_multi_problem_ctas_and_sub_batches(env):
    """400 cells x 12 months at n = 145..168 (NB 19-21): each CTA solves many problems, with the software pipeline and
    the deferred trend solve of the previous problem.  Interleaved: two points that see a co-located station pair
    (TWXI_ST_SINGULAR), n = 1, 3, 4 (TWXI_ST_SINGULAR) and n = 169, 200, 255 (TWXI_ST_LIMIT).  Bitwise equal to the same
    batch with TWXI_HC_BUDGET_MB=0 (one point per staging sub-batch, one problem per CTA); a sample against ked_exact."""
    db = env["db"]
    s = env["da"].stns.copy()
    good = np.flatnonzero(env["mask"])
    plat, plon, _, _ = _cells(env, [5], [5])
    a, b = good[env["nbrs"](plat[0], plon[0], 2)]
    s[db.LON][b], s[db.LAT][b] = s[db.LON][a], s[db.LAT][a]
    da = db.StationSerialDataDb((s, env["da"].var, env["da"].days), env["da"].var_name)
    ctx = _ctx(env, da)
    rr, cc = np.meshgrid(np.arange(215, 235), np.arange(215, 235), indexing="ij")
    blat, blon, belev, blst = _cells(env, rr.ravel(), cc.ravel())
    rng = np.random.default_rng(19)
    bnn = rng.integers(145, MAX_N + 1, blat.size).astype(np.int32)
    bvo = np.column_stack([rng.uniform(0.05, 0.5, blat.size), rng.uniform(0.5, 2.0, blat.size),
                           rng.uniform(20.0, 300.0, blat.size)])
    flat, flon, felev, flst = _cells(env, [5, 6, 214, 214, 214, 235, 235, 235], [5, 4, 214, 220, 230, 214, 220, 230])
    fnn = np.array([40, 40, 1, 3, 4, 169, 200, 255], dtype=np.int32)
    fst = [ST_SINGULAR] * 5 + [ST_LIMIT] * 3
    fat = [0, 50, 101, 163, 222, 287, 350, 407]                      # batch rows of the failing points
    n = blat.size + flat.size
    isf = np.zeros(n, dtype=bool)
    isf[fat] = True

    def place(bv, fv):
        out = np.empty((n,) + bv.shape[1:], dtype=bv.dtype)
        out[~isf], out[isf] = bv, fv
        return out
    lat, lon, elev, lst = place(blat, flat), place(blon, flon), place(belev, felev), place(blst, flst)
    nn, vo = place(bnn, fnn), place(bvo, np.tile([0.2, 1.1, 120.0], (flat.size, 1)))
    mean, var, st = ctx.krig(lat, lon, elev, lst, mth=0, nnghs=nn, vario=vo)
    assert np.array_equal(st[isf], fst), st[isf]
    assert np.all(st[~isf] == ST_OK)
    old = os.environ.get("TWXI_HC_BUDGET_MB")
    os.environ["TWXI_HC_BUDGET_MB"] = "0"
    try:
        mean1, var1, st1 = ctx.krig(lat, lon, elev, lst, mth=0, nnghs=nn, vario=vo)
    finally:
        if old is None:
            os.environ.pop("TWXI_HC_BUDGET_MB", None)
        else:
            os.environ["TWXI_HC_BUDGET_MB"] = old
    assert np.array_equal(st, st1)
    assert np.array_equal(mean[~isf], mean1[~isf]) and np.array_equal(var[~isf], var1[~isf])
    # the exact reference on a sample of the cells (their neighbours from the library's kNN on the modified table)
    rows = np.flatnonzero(~isf)[rng.choice(blat.size, 16, replace=False)]
    idx, _, _, kst = ctx.knn(lat[rows], lon[rows], MAX_N)
    assert np.all(kst == 0)
    probs, at = [], []
    for j, r in enumerate(rows):
        m = int(rng.integers(1, 13))
        probs.append(dict(gid=j, pt=(lon[r], lat[r], elev[r], lst[r, m - 1]), sids=idx[j, :nn[r]], mth=m,
                          vario=tuple(vo[r])))
        at.append((r, m))
    ref, _ = reference(s[np.isnan(s[db.BAD])], probs)
    stats, bad = _Stats(), []
    for (r, m), rf in zip(at, ref):
        _check(stats, "many problems per CTA", rf, mean[r, m - 1], var[r, m - 1], bad, (r, m, nn[r]))
    stats.report("D. multi-problem CTAs against ked_exact")
    assert not bad, (len(bad), bad[:10])


# ---- E. covariance domain -------------------------------------------------------------------------------------------
def ols_exact(X, y, x0, c00):
    """Closed-form OLS at DPS digits: the kriging predictor of the pure nugget model V = C(0) I.
    mean = x0'b, b = (X'X)^-1 X'y;  var = C(0) (1 + x0'(X'X)^-1 x0)  (X, x0 with the intercept, uncentred)."""
    with mpmath.workdps(DPS):
        A = mpmath.matrix([[mpmath.mpf(1)] + [_mp(v) for v in row] for row in np.asarray(X)])
        f0 = mpmath.matrix([mpmath.mpf(1)] + [_mp(v) for v in x0])
        G = A.T * A
        b = mpmath.lu_solve(G, A.T * mpmath.matrix([_mp(v) for v in y]))
        g = mpmath.lu_solve(G, f0)
        return (f0.T * b)[0], _mp(c00) * (1 + (f0.T * g)[0])


@pytest.mark.gpu
def test_covariance_domain_vs_exact(env, case_e):
    """Pure nugget (range 0, psill 0: also against closed-form OLS), nugget 0, a 3 m range (-1/range clamped at
    -250/km), a 50 m range (covariances below 2^-1000), prediction at a station without rm_zero (the mean is the
    station's normal, the variance 0, each within its bound) and next to a station (the variance carries one covariance
    at f = -0.499: a covariance error of 3e-14 relative shows there): one call, within the bounds."""
    from topowx_b200 import db
    c = case_e
    ctx = _ctx(env)
    q = np.array([p[0] for p in c["pts"]])
    nn = np.array([p[1] for p in c["pts"]], dtype=np.int32)
    vo = np.array([c["varios"][p[2]] for p in c["pts"]])
    mean, var, st = ctx.krig(c["lat"][q], c["lon"][q], c["elev"][q], c["lst"][q], mth=MTH_A, nnghs=nn, vario=vo)
    assert np.all(st == ST_OK)
    stats, bad = _Stats(), []
    s = env["stns"]
    for b, (qq, n, v) in enumerate(c["pts"]):
        ref = c["ref"][b]
        _check(stats, v, ref, mean[b, 0], var[b, 0], bad, (qq, n, v))
        if v.startswith("pure nugget"):
            sids = env["nbrs"](c["lat"][qq], c["lon"][qq], n)
            X = np.column_stack([s[db.LON][sids], s[db.LAT][sids], s[db.ELEV][sids],
                                 s[db.get_lst_varname(MTH_A)][sids]])
            x0 = (c["lon"][qq], c["lat"][qq], c["elev"][qq], c["lst"][qq, MTH_A - 1])
            om, ov = ols_exact(X, s[db.get_norm_varname(MTH_A)][sids], x0, sum(c["varios"][v][:2]))
            _check(stats, v + " vs OLS", dict(ref, mean=om, var=ov), mean[b, 0], var[b, 0], bad, (qq, n, v, "OLS"))
        if qq in (2, 3):
            j = c["on"][qq - 2]
            assert abs(mean[b, 0] - s[db.get_norm_varname(MTH_A)][j]) <= ref["mean_bound"], (qq, n, v)
            assert abs(var[b, 0]) <= ref["var_bound"], (qq, n, v)
    stats.report("E. covariance domain against ked_exact")
    assert not bad, (len(bad), bad[:10])


# ---- F. fewer than 5 neighbours -------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_fewer_than_five_neighbours_is_singular(env, case_f):
    """n = 1..4 (fewer neighbours than the five trend coefficients): TWXI_ST_SINGULAR for exactly those points of a
    mixed batch; n = 5 and 6 are computed, within their bounds."""
    c = case_f
    ctx = _ctx(env)
    counts = (1, 2, 3, 4, 5, 6)
    q = np.repeat(np.arange(c["lat"].size), len(counts))
    nn = np.tile(np.asarray(counts, dtype=np.int32), c["lat"].size)
    mean, var, st = ctx.krig(c["lat"][q], c["lon"][q], c["elev"][q], c["lst"][q], mth=MTH_A, nnghs=nn,
                             vario=VARIOS["typical"])
    assert np.array_equal(st, np.where(nn < 5, ST_SINGULAR, ST_OK)), st
    stats, bad = _Stats(), []
    for b in np.flatnonzero(nn >= 5):
        ref = c["ref"][2 * q[b] + (nn[b] - 5)]
        _check(stats, "n = %d" % nn[b], ref, mean[b, 0], var[b, 0], bad, (q[b], nn[b]))
    stats.report("F. n = 5, 6 against ked_exact")
    assert not bad, (len(bad), bad[:10])


# ---- the reference itself (CPU) -------------------------------------------------------------------------------------
def _random_case(seed, n):
    """A random neighbourhood in the style of test_oracle_ked._case; the point is no station."""
    r = np.random.default_rng(seed)
    lon, lat = r.uniform(-101, -97, n), r.uniform(38, 43, n)
    elev, lst = r.uniform(200, 2500, n), r.normal(10, 6, n)
    X = np.column_stack([lon, lat, elev, lst])
    y = 12 - 0.005 * elev - 0.5 * (lat - 40) + 0.2 * lst + r.normal(0, 0.7, n)
    return X, y, np.array([-99.1, 40.4, 950.0, 11.0])


def _exact_of(X, y, x0, vario, keep=False):
    with mpmath.workdps(DPS):
        n = len(y)
        H = [[gcdist_exact(X[i, 0], X[i, 1], X[j, 0], X[j, 1]) if i != j else mpmath.mpf(0) for j in range(n)]
             for i in range(n)]
        h0 = [gcdist_exact(x0[0], x0[1], X[j, 0], X[j, 1]) for j in range(n)]
        return ked_exact(X, y, x0, vario, H, h0, keep)


@pytest.mark.parametrize("n", [5, 8, 40])
@pytest.mark.parametrize("vario", ["typical", "long range"])
def test_exact_matches_oracle_within_float64_bound(n, vario):
    """ked_exact against the float64 oracle (ked_gstat: GLS form, Cholesky, drift scaled by its largest value)."""
    X, y, x0 = _random_case(n, n)
    r = _exact_of(X, y, x0, VARIOS[vario])
    om, ov = o.ked_gstat(X[:, 0], X[:, 1], X, y, x0[0], x0[1], x0, *VARIOS[vario])
    assert r["converged"]
    assert abs(float(r["mean"] - _mp(om))) <= r["mean_bound"], (float(r["mean"]), om, r["mean_bound"])
    assert abs(float(r["var"] - _mp(ov))) <= r["var_bound"], (float(r["var"]), ov, r["var_bound"])


def test_exact_weights_satisfy_the_drift_constraints():
    """F'lambda = f0 (the unbiasedness conditions of universal kriging) to 1e-30, uncentred drift."""
    for n, v in ((5, "typical"), (33, "short range"), (90, "long range")):
        X, y, x0 = _random_case(100 + n, n)
        r = _exact_of(X, y, x0, VARIOS[v], keep=True)
        assert r["converged"]
        with mpmath.workdps(DPS):
            for a in range(5):
                e = mpmath.fdot(r["lam"], r["F"][:, a]) - r["f0"][a]
                assert abs(e) <= 1e-30 * max(1, abs(r["f0"][a])), (n, v, a, e)


def test_exact_pure_nugget_is_ols():
    """V = C(0) I for range 0 and for psill 0: ked_exact equals closed-form OLS to 1e-30."""
    X, y, x0 = _random_case(3, 30)
    for vario in ((0.4, 0.9, 0.0), (1.3, 0.0, 80.0)):
        r = _exact_of(X, y, x0, vario)
        om, ov = ols_exact(X, y, x0, vario[0] + vario[1])
        assert abs(r["mean"] - om) <= 1e-30 * abs(om) and abs(r["var"] - ov) <= 1e-30 * abs(ov), vario


def test_exact_reproduces_the_value_at_a_station():
    """Prediction at a station (distance exactly 0, covariance C(0)): the station's value, variance 0, to 1e-30."""
    X, y, _ = _random_case(4, 25)
    j = 6
    for v in ("typical", "long range"):
        r = _exact_of(X, y, X[j], VARIOS[v])
        assert abs(r["mean"] - _mp(y[j])) <= 1e-30 and abs(r["var"]) <= 1e-30, v


def test_refinement_converges_on_every_gpu_case(case_a, case_e, case_f):
    """Iterative refinement reaches 1e-35 on every problem of cases A, C (= A), E and F without the mpmath.lu_solve
    fallback; B and D check it on their problems as they run."""
    steps = []
    for c in (case_a, case_e, case_f):
        for r in c["ref"]:
            assert r["converged"]
            steps.append(r["steps"])
    print("refinement steps: max %d, mean %.2f over %d problems" % (max(steps), np.mean(steps), len(steps)))


def test_host_distance_error_fits_c_h(case_a):
    """numpy's float64 gcdist_sp against gcdist_exact on every pair of case A: within C_H / 4 eps relative (the rest of
    C_H is the device's larger trig error and a margin, see C_H)."""
    p = np.array(case_a["dist"]["pairs"])
    ex = case_a["dist"]["dist"]
    h = o.gcdist_sp(p[:, 0], p[:, 1], p[:, 2], p[:, 3])
    worst = max(abs(float((_mp(a) - e) / e)) for a, e in zip(h, ex) if e != 0) / EPS
    print("float64 gcdist_sp: worst relative error %.2f eps over %d pairs" % (worst, len(ex)))
    assert worst <= C_H / 4


def test_oracle_reports_fewer_than_five_neighbours_as_singular():
    """ked_gstat raises ST_SINGULAR for n = 1..4 whatever the rounded factorisations say, and solves n = 5."""
    for n in (1, 2, 3, 4):
        for seed in range(50):
            X, y, x0 = _random_case(1000 * n + seed, n)
            with pytest.raises(o.OracleError) as e:
                o.ked_gstat(X[:, 0], X[:, 1], X, y, x0[0], x0[1], x0, *VARIOS["typical"])
            assert e.value.status == o.ST_SINGULAR
    X, y, x0 = _random_case(5, 5)
    mean, var = o.ked_gstat(X[:, 0], X[:, 1], X, y, x0[0], x0[1], x0, *VARIOS["typical"])
    assert np.isfinite(mean) and np.isfinite(var)

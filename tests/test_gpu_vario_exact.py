"""vario_fit_kernel (twxi_fit_vario, twxi_krig_all) against a 40-digit restatement of its five stages.

The float64 oracle runs the same algorithm as the kernel, so an algorithmic error they share cancels in
test_variogram_fit_and_krig_all_vs_oracle.  The referee here is ``vario_exact``: OLS residuals, exact lag sums, the range
as the root of dS/dr (Gauss-Newton path, then Newton to 1e-30), GLS through a 40-digit Cholesky and the second fit, with
the kernel's float64 inputs taken as exact.  Each tolerance comes from the problem's own conditioning, computed by the
reference (see ``_range_bound``), so a kernel that stops the range fit short, coarsens the fixed-point lag sums, mixes the
two variograms or builds V wrongly fails.

Counts cover n = 6 (TWXI_ST_SINGULAR), 7, the warp (32) and CTA (256 threads; 8 warps) strides, and n = 168
(TWXI_MAX_KRIG_NNGHS) and 169 (TWXI_ST_LIMIT); a sparse CONUS table gives hundreds of lags on both sides of the 512-lag
limit.  Run with -m gpu; the reference's own checks at the end run on the CPU."""
import multiprocessing as mp
import os

import numpy as np
import pytest

mpmath = pytest.importorskip("mpmath")      # comes with torch (through sympy)

from oracle import twx_oracle as o          # noqa: E402

DPS = 40
EPS = 2.0 ** -53
C_BOUND = 64
G_FLOOR = 2.0 ** -37                        # vario.cu VF_GSCALE = 2^36: half a unit of the squared-difference grid
H_FLOOR = 2.0 ** -31                        # vario.cu VF_HSCALE = 2^30: half a unit of the distance grid
WIDTH, MAXBIN, MAX_N = 5.0, 512, 168
COUNTS = [6, 7, 8, 9, 15, 16, 17, 31, 32, 33, 63, 64, 65, 100, 127, 128, 129, 147, 167, 168, 169]
BIG_MONTHS = (1, 4, 7, 12)                  # months compared above n = 65 (all 12 at n <= 65)
ST_OK, ST_SINGULAR, ST_LIMIT = 0, 4, 8
IDENT_CURV, IDENT_EXP = 1e-8, 1e-12


# ---- the reference --------------------------------------------------------------------------------------------------
def _mp(x):
    return mpmath.mpf(float(x))


def _solve(A, b):
    """Gaussian elimination with partial pivoting (5x5, working precision)."""
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


def _lstsq(cols, rhs):
    """beta of min |rhs - sum beta_c cols_c| by the normal equations (exact data, working precision)."""
    A = [[mpmath.fdot(a, b) for b in cols] for a in cols]
    return _solve(A, [mpmath.fdot(a, rhs) for a in cols])


def _sill(z):
    n = len(z)
    m = mpmath.fsum(z) / n
    return mpmath.fsum((t - m) ** 2 for t in z) / (n - 1)


def _variogram(pi, pj, hk, lag, z):
    """Exact lag sums of the kept pairs: per non-empty lag in lag order (np, mean h, gamma = sum dz^2 / 2 np)."""
    acc = {}
    for i, j, h, b in zip(pi, pj, hk, lag):
        d = z[i] - z[j]
        a = acc.setdefault(b, [0, [], []])
        a[0] += 1
        a[1].append(h)
        a[2].append(d * d)
    keys = sorted(acc)
    cnt = [acc[b][0] for b in keys]
    hs = [mpmath.fsum(_mp(h) for h in acc[b][1]) / acc[b][0] for b in keys]
    gs = [mpmath.fsum(acc[b][2]) / (2 * acc[b][0]) for b in keys]
    return cnt, hs, gs


def _terms(cnt, hs, gs, nug, ps, r):
    """S(r) = sum w e^2, g(r) = sum w J e (dS/dr = -2 g), g'(r), den = sum w J^2 (w = np / h^2, J = d model / d r)."""
    S = g = gp = den = 0
    for c, h, gm in zip(cnt, hs, gs):
        w = c / (h * h)
        ex = mpmath.exp(-h / r)
        e = gm - (nug + ps * (1 - ex))
        J = -ps * ex * h / (r * r)
        dJ = ps * ex * h * (2 * r - h) / r ** 4
        S += w * e * e
        g += w * J * e
        gp += w * (dJ * e - J * J)
        den += w * J * J
    return S, g, gp, den


def _fit(cnt, hs, gs, sill):
    """Stage 3: nugget = min gamma, psill = sill - nugget, range = the root of dS/dr reached by the damped Gauss-Newton
    path of vario.cu from 0.1 max h, polished by Newton to 1e-30.  branch: 'psill<0', 'den<=0', 'noroot' or 'range'."""
    nug = min(gs)
    ps = sill - nug
    out = dict(K=len(cnt), nug=nug, ps=ps, r=mpmath.mpf(0), first_step=None)
    if ps < 0:
        return dict(out, branch="psill<0")
    if ps == 0:
        return dict(out, branch="den<=0")
    sse = lambda r: _terms(cnt, hs, gs, nug, ps, r)[0]
    r = hs[-1] / 10
    s_old = sse(r)
    for it in range(400):
        _, g, _, den = _terms(cnt, hs, gs, nug, ps, r)
        if not den > 0:
            return dict(out, branch="den<=0")
        step, found = g / den, False
        for _h in range(12):
            rn = r + step
            if rn > 0:
                s_new = sse(rn)
                if s_new <= s_old:
                    found = True
                    break
            step /= 2
        if it == 0:
            out["first_step"] = found
        if not found:
            break
        r, s_old = rn, s_new
        if abs(step) <= mpmath.mpf(10) ** -12 * r:
            break
    for _it in range(60):
        _, g, gp, _ = _terms(cnt, hs, gs, nug, ps, r)
        if not gp < 0 or not r > 0:
            break
        step = -g / gp
        r += step
        if abs(step) <= mpmath.mpf(10) ** -32 * r:
            break
    S, g, gp, _ = _terms(cnt, hs, gs, nug, ps, r)
    if not (r > 0 and gp < 0 and abs(g) * r <= mpmath.mpf(10) ** -28 * S):
        return dict(out, branch="noroot", r=r)
    # not identifiable: S flat in r (S'' r^2 / S tiny) or the model is the sill at every lag (range far below them)
    small = mpmath.exp(-hs[0] / r) < IDENT_EXP
    flat = -2 * gp * r * r / S < IDENT_CURV
    return dict(out, branch="range", r=r, S=S, g=g, gp=gp, ident=not (small or flat), small=bool(small))


def _range_bound(cnt, hs, gs, nug, ps, r, gp, dg, dh, dn, ds):
    """|dr*/dtheta| dtheta summed over theta = every gamma_k, mean distance h_k, the nugget and the sill, with
    dr*/dtheta = -(dg/dtheta) / g'(r*) (implicit function theorem, exact), plus the root error of a float64 Newton
    step: the rounding of g itself, C eps sum |w J| (|gamma| + nugget + psill), over |g'|."""
    sill = nug + ps
    acc_g = acc_h = d_n = d_s = rnd = 0
    for k, (c, h, gm) in enumerate(zip(cnt, hs, gs)):
        w = c / (h * h)
        ex = mpmath.exp(-h / r)
        e = gm - sill + ps * ex
        J = -ps * ex * h / (r * r)
        acc_g += abs(w * J) * dg[k]
        dw = -2 * c / h ** 3
        dJh = -ps * ex * (1 - h / r) / (r * r)
        de = -ps * ex / r
        acc_h += abs(dw * J * e + w * dJh * e + w * J * de) * dh[k]
        d_n += w * (ex * h / (r * r) * e - J * ex)
        d_s += w * (-ex * h / (r * r) * e + J * (ex - 1))
        rnd += abs(w * J) * (abs(gm) + sill)
    tot = acc_g + acc_h + abs(d_n) * dn + abs(d_s) * ds + C_BOUND * EPS * rnd
    return tot / abs(gp), dict(gamma=float(acc_g / abs(gp)), dist=float(acc_h / abs(gp)),
                               nugget=float(abs(d_n) * dn / abs(gp)), sill=float(abs(d_s) * ds / abs(gp)),
                               rounding=float(C_BOUND * EPS * rnd / abs(gp)))


def _deltas(cnt, hs, gs, sill, dz):
    """Errors of the kernel's lag means and sill: the float64 sums, the fixed-point grids, and residual errors dz carried
    through gamma = mean dz^2 / 2 (|d gamma| <= 2 dz sqrt(2 gamma))."""
    dg = [C_BOUND * EPS * g + G_FLOOR + 2 * dz * mpmath.sqrt(2 * g) for g in gs]
    dh = [C_BOUND * EPS * h + H_FLOOR for h in hs]
    ds = C_BOUND * EPS * sill + 2 * dz * mpmath.sqrt(2 * sill)
    return dg, dh, max(dg), ds


def _kappa(A):
    """cond_2 of the symmetric matrix A with its diagonal scaled to 1: a Cholesky-based solve does not see the column
    scaling (van der Sluis), so this is the condition that its rounding is amplified by."""
    d = np.sqrt(np.diag(A))
    return float(np.linalg.cond(A / d[:, None] / d[None, :]))


def _kernel_X(lon, lat, elev, lst):
    """The kernel's predictors: centred on the nearest neighbour, elevation in km, lst / 10 (float64, as vario.cu)."""
    return np.column_stack([np.ones(lon.size), lon - lon[0], lat - lat[0], (elev - elev[0]) * 1e-3, (lst - lst[0]) * 0.1])


def _stage5_f64(H, X, y, cutoff, model):
    """Stages 4-5 in float64 (the oracle's algorithm) for a given first model: (nugget, psill, range) of the output."""
    nug, ps, r = model
    n = y.size
    V = ps * np.exp(-H / r)
    V[np.diag_indices(n)] = nug + ps
    Lc = np.linalg.cholesky(V)
    Z = np.linalg.solve(Lc, np.column_stack((X, y)))
    beta = np.linalg.solve(Z[:, :-1].T @ Z[:, :-1], Z[:, :-1].T @ Z[:, -1])
    z = y - X @ beta
    sill = float(np.var(z, ddof=1))
    npairs, dist, gamma = o.sample_variogram(H, z, cutoff)
    m = o.fit_exp_range(npairs, dist, gamma, float(np.min(gamma)), sill)
    return np.array([sill, 0.0, 0.0]) if m is None else np.array(m)


def vario_exact(lon, lat, elev, lst, y, dmax):
    """The variogram of one neighbourhood (neighbours in kNN order, dmax = the library's distance of the last one).

    Returns dict(status, nb, near, branch1, branch2, out (nugget, psill, range) rounded once, bound (3), ident, small,
    plus diagnostics).  Status ST_SINGULAR for n < 7 or a zero pair distance, ST_LIMIT for more than 512 lags."""
    lon, lat, elev, lst, y = (np.asarray(a, dtype=np.float64) for a in (lon, lat, elev, lst, y))
    n = y.size
    if n < 7:
        return dict(status=ST_SINGULAR, why="n<7")
    if n > MAX_N:
        return dict(status=ST_LIMIT, why="n>%d" % MAX_N)
    H = o.gcdist_sp(lon[:, None], lat[:, None], lon[None, :], lat[None, :])
    pi, pj = np.triu_indices(n, 1)
    h = H[pi, pj]
    if np.any(h == 0.0):
        return dict(status=ST_SINGULAR, why="colocated")
    cutoff = float(dmax) * 1.4
    nb = int(np.floor(cutoff / WIDTH)) + 1
    if nb > MAXBIN:
        return dict(status=ST_LIMIT, nb=nb)
    keep = h <= cutoff
    lag = np.floor(h / WIDTH).astype(np.int64)
    # pairs whose lag or cutoff decision a last-ulp difference of the device's libm could flip
    bnd = WIDTH * np.round(h / WIDTH)
    near = int(np.sum((np.abs(h - bnd) <= 1e-12 * h) & (bnd > 0)) + np.sum(np.abs(h - cutoff) <= 1e-12 * cutoff))
    pi, pj, hk, lag = pi[keep], pj[keep], h[keep], lag[keep]
    X = _kernel_X(lon, lat, elev, lst)
    kap1 = _kappa(X.T @ X)
    ymax = float(np.abs(y).max())
    res = dict(status=ST_OK, nb=nb, near=near, n=n)
    with mpmath.workdps(DPS):
        one = mpmath.mpf(1)
        cols = [[one] * n] + [[_mp(a) - _mp(v[0]) for a in v] for v in (lon, lat, elev, lst)]
        Y = [_mp(t) for t in y]
        b1 = _lstsq(cols, Y)
        z1 = [Y[j] - mpmath.fsum(b1[c] * cols[c][j] for c in range(5)) for j in range(n)]
        sill1 = _sill(z1)
        c1, h1, g1 = _variogram(pi, pj, hk, lag, z1)
        f1 = _fit(c1, h1, g1, sill1)
        dz1 = C_BOUND * EPS * kap1 * ymax
        res.update(branch1=f1["branch"], K=f1["K"], first_step=f1["first_step"], ident1=f1.get("ident"),
                   sill1=float(sill1), nug1=float(f1["nug"]), r1=float(f1["r"]), dz1=dz1)
        dg1, dh1, dn1, ds1 = _deltas(c1, h1, g1, sill1, dz1)
        res["psill1_margin"] = float(abs(f1["ps"]) / (dn1 + ds1))
        if f1["branch"] == "range":
            dr1, _ = _range_bound(c1, h1, g1, f1["nug"], f1["ps"], f1["r"], f1["gp"], dg1, dh1, dn1, ds1)
            res["dr1"] = float(dr1)
            nug, ps, r = f1["nug"], f1["ps"], f1["r"]
            V = [[(nug + ps) if i == j else ps * mpmath.exp(-_mp(H[i, j]) / r) for j in range(i + 1)] for i in range(n)]
            L = [[None] * (i + 1) for i in range(n)]
            for i in range(n):
                Li = L[i]
                for j in range(i + 1):
                    s = V[i][j] - (mpmath.fdot(Li[:j], L[j][:j]) if j else 0)
                    if i == j:
                        if not s > 0:
                            return dict(res, status=ST_SINGULAR, why="cholesky")
                        Li[i] = mpmath.sqrt(s)
                    else:
                        Li[j] = s / L[j][j]

            def fwd(v):
                out = []
                for i in range(n):
                    out.append((v[i] - (mpmath.fdot(L[i][:i], out) if i else 0)) / L[i][i])
                return out
            zc = [fwd(c) for c in cols]
            b2 = _lstsq(zc, fwd(Y))
            z2 = [Y[j] - mpmath.fsum(b2[c] * cols[c][j] for c in range(5)) for j in range(n)]
            Vf = np.array([[float(V[max(i, j)][min(i, j)]) for j in range(n)] for i in range(n)])
            Lf = np.linalg.cholesky(Vf)
            Zf = np.linalg.solve(Lf, X)
            kap2 = _kappa(Vf) + _kappa(Zf.T @ Zf)
            dz2 = C_BOUND * EPS * kap2 * ymax
            if f1["ident"]:
                # stages 4-5 against the first range: central difference of the float64 pipeline (it only needs a few
                # correct digits, since it multiplies dr1)
                m0 = (float(nug), float(ps), float(r))
                step = 1e-6 * m0[2]
                dp = _stage5_f64(H, X, y, cutoff, (m0[0], m0[1], m0[2] + step))
                dm = _stage5_f64(H, X, y, cutoff, (m0[0], m0[1], m0[2] - step))
                d_r1 = np.abs(dp - dm) / (2 * step) * float(dr1)
            else:
                d_r1 = None
        else:
            # pure nugget: V = sill I, GLS = OLS.  Without a minimum in r the kernel still has some range and runs the
            # GLS with it, so its stage 5 is not defined by the data: not compared
            z2, dz2, d_r1 = z1, dz1, (None if f1["branch"] == "noroot" else np.zeros(3))
        sill2 = _sill(z2)
        c2, h2, g2 = _variogram(pi, pj, hk, lag, z2)
        f2 = _fit(c2, h2, g2, sill2)
        dg2, dh2, dn2, ds2 = _deltas(c2, h2, g2, sill2, dz2)
        res.update(branch2=f2["branch"], dz2=dz2, ident=f2.get("ident"), small=f2.get("small"),
                   psill2_margin=float(abs(f2["ps"]) / (dn2 + ds2)), stage5_comparable=d_r1 is not None)
        if f2["branch"] == "range":
            dr2, terms = _range_bound(c2, h2, g2, f2["nug"], f2["ps"], f2["r"], f2["gp"], dg2, dh2, dn2, ds2)
            res["out"] = np.array([float(f2["nug"]), float(f2["ps"]), float(f2["r"])])
            bound = np.array([float(dn2), float(dn2 + ds2), float(dr2)])
            res["range_terms"] = terms
            res["S2"], res["g2"], res["gp2"] = float(f2["S"]), float(f2["g"]), float(f2["gp"])
        elif f2["branch"] == "noroot":                  # S has no minimum in r: only nugget and psill are defined
            res["out"] = np.array([float(f2["nug"]), float(f2["ps"]), np.inf])
            bound = np.array([float(dn2), float(dn2 + ds2), np.inf])
            res["sill2"], res["dsill2"] = float(sill2), float(ds2)
        else:
            res["out"] = np.array([float(sill2), 0.0, 0.0])
            bound = np.array([float(ds2), 0.0, 0.0])
        res["bound"] = bound + (0.0 if d_r1 is None else d_r1)
        res["d_r1"] = d_r1
        res["h0"] = float(h2[0])
    return res


def _ref_task(args):
    return vario_exact(*args)


def _farm(tasks):
    """vario_exact over every host core (fork pool, as oracle/cpu_farm.py)."""
    n = max(1, os.cpu_count() or 1)
    with mp.get_context("fork").Pool(n) as pool:
        return pool.map(_ref_task, tasks, chunksize=1)


# ---- comparison -----------------------------------------------------------------------------------------------------
class _Stats(object):
    """Worst error / bound per (quantity, layout, count class), and the loosest range bounds."""

    def __init__(self):
        self.d, self.loose, self.branches = {}, [], {}

    def add(self, key, ratio):
        self.d[key] = max(self.d.get(key, 0.0), float(ratio))

    def report(self, title):
        print("\n" + title)
        for key in sorted(self.d):
            print("  %-40s worst error/bound %.3g" % (" ".join(map(str, key)), self.d[key]))
        print("  branches (first fit, second fit): %s" % sorted((str(k), c) for k, c in self.branches.items()))
        for w in sorted(self.loose, key=lambda t: -t[1])[:8]:
            print("  range bound looser than 1e-10 relative: %s  bound/range %.3g  dominant %s" % w)


def _cls(n):
    return "n<=33" if n <= 33 else ("n<=65" if n <= 65 else "n>=100")


def _compare(stats, bad, layout, key, got, st, ref):
    """One (point, month) of the kernel against vario_exact."""
    stats.branches[ref.get("branch1"), ref.get("branch2")] = stats.branches.get((ref.get("branch1"),
                                                                                 ref.get("branch2")), 0) + 1
    if ref["status"] != ST_OK:
        if st != ref["status"]:
            bad.append((layout, key, "status", st, ref["status"]))
        elif not np.all(np.isnan(got)):
            bad.append((layout, key, "failed point not NaN", got))
        return
    if st != ST_OK:
        bad.append((layout, key, "status", st, ref))
        return
    if ref["near"] or not ref["stage5_comparable"] or ref["psill1_margin"] < 1 or ref["psill2_margin"] < 1:
        stats.add(("skipped: lag boundary / unidentifiable first range / psill ~ 0", layout, "count"), 1)
        return
    cls = _cls(ref["n"])
    out, bound = ref["out"], ref["bound"]
    err = np.abs(got - out)
    if ref["branch2"] == "noroot" and got[2] == 0.0:    # the float64 path ended without a range: pure nugget
        ref = dict(ref, out=np.array([ref["sill2"], 0.0, 0.0]), bound=np.array([ref["dsill2"], 0.0, 0.0]),
                   branch2="noroot -> pure nugget")
        out, bound = ref["out"], ref["bound"]
        err = np.abs(got - out)
    if ref["branch2"] not in ("range", "noroot"):
        stats.add(("pure nugget sill (%s)" % ref["branch2"], layout, cls), err[0] / bound[0])
        if err[0] > bound[0] or got[1] != 0.0 or got[2] != 0.0:
            bad.append((layout, key, "pure nugget", got, out, bound))
        return
    for c, what in ((0, "nugget"), (1, "psill")):
        stats.add((what, layout, cls), err[c] / bound[c])
        if err[c] > bound[c]:
            bad.append((layout, key, what, got, out, bound))
    if ref["branch2"] == "noroot":
        stats.add(("range not compared: no minimum in r", layout, cls), 1)
    elif ref["ident"]:
        stats.add(("range", layout, cls), err[2] / bound[2])
        if err[2] > bound[2]:
            bad.append((layout, key, "range", got, out, bound, ref["range_terms"]))
        if bound[2] > 1e-10 * out[2]:
            t = ref["range_terms"]
            stats.loose.append((str(key), bound[2] / out[2], max(t, key=t.get)))
    elif ref["small"]:
        stats.add(("range below the lags: range < h0/30", layout, cls), got[2] / (ref["h0"] / 30))
        if not got[2] < ref["h0"] / 30:
            bad.append((layout, key, "unidentifiable range", got, out))


# ---- fixtures -------------------------------------------------------------------------------------------------------
def _arrays(d, gidx, m):
    from topowx_b200 import db
    s = d.stns[gidx]
    return (s[db.LON], s[db.LAT], s[db.ELEV], s[db.get_lst_varname(m)], s[db.get_norm_varname(m)])


def _tasks(d, gidx, dist, counts_months):
    """vario_exact tasks of (point q, count n, month m) for the kNN rows gidx / dist."""
    tasks, meta = [], []
    for q, n, m in counts_months:
        tasks.append(_arrays(d, gidx[q, :n], m) + (dist[q, n - 1],))
        meta.append((q, n, m))
    return tasks, meta


@pytest.fixture(scope="module")
def dense():
    """Fixture A: ~3200 stations over the tile bbox, both variables; 6 tile cells, 3 stations queried without rm_zero
    (the station is its own neighbour at d = 0, step 22) and 3 with rm_zero (XvalTairNorm)."""
    from topowx_b200 import synth, db
    from topowx_b200.context import TwxiContext
    f = synth.Fields()
    days = synth.make_days(1995, 1)
    rng = np.random.default_rng(20261021)
    rows = rng.integers(synth.TILE_ROW0 + 20, synth.TILE_ROW0 + synth.TILE_SIZE - 20, 6)
    cols = rng.integers(synth.TILE_COL0 + 20, synth.TILE_COL0 + synth.TILE_SIZE - 20, 6)
    out = []
    for w in (0, 1):
        d = synth.make_station_db(w, 3200, synth.tile_bbox(), f, days)
        ctx = TwxiContext(d, np.isnan(d.stns[db.BAD]))
        good = ctx.gidx[np.isfinite(d.stns[db.MASK][ctx.gidx])]
        stn = good[rng.choice(good.size, 6, replace=False)]
        lat = np.concatenate([synth.grid_lats(rows), d.stns[db.LAT][stn]])
        lon = np.concatenate([synth.grid_lons(cols), d.stns[db.LON][stn]])
        rmz = np.array([False] * 9 + [True] * 3)
        groups = []
        for sel, z in ((~rmz, False), (rmz, True)):
            idx, dist, _, st = ctx.knn(lat[sel], lon[sel], max(COUNTS), rm_zero=z)
            assert np.all(st == 0)
            groups.append((np.flatnonzero(sel), ctx.gidx[idx], dist, z))
        gidx = np.zeros((lat.size, max(COUNTS) + 1), dtype=np.int64)
        dist = np.zeros((lat.size, max(COUNTS) + 1))
        for sel, gi, di, _ in groups:
            gidx[sel], dist[sel] = gi, di
        assert np.all(dist[6:9, 0] == 0.0) and np.all(dist[9:, 0] > 0.0)
        cm = [(q, n, m) for q in range(lat.size) for n in COUNTS
              for m in (range(1, 13) if n <= 65 else BIG_MONTHS)]
        tasks, meta = _tasks(d, gidx, dist, cm)
        ref = dict(zip(meta, _farm(tasks)))
        out.append(dict(d=d, ctx=ctx, lat=lat, lon=lon, rmz=rmz, gidx=gidx, dist=dist, ref=ref, f=f, w=w))
    return out


def _fit_batch(v, sel, counts, mth=0):
    """fit_vario of points ``sel`` x ``counts`` as one batch: point i, count c at row i * len(counts) + c."""
    nc = len(counts)
    lat, lon = np.repeat(v["lat"][sel], nc), np.repeat(v["lon"][sel], nc)
    nn = np.tile(np.asarray(counts, dtype=np.int32), len(sel))
    z = bool(v["rmz"][sel[0]])
    assert np.all(v["rmz"][sel] == z)
    return v["ctx"].fit_vario(lat, lon, mth=mth, nnghs=nn, rm_zero=z)


# ---- 1. dense table: every count, every stage ----------------------------------------------------------------------
@pytest.mark.gpu
def test_fit_vario_dense_vs_exact(dense):
    """fit_vario of 12 points x 21 counts x 12 months, both variables, in one batch per (variable, rm_zero) against
    vario_exact; n = 6 is TWXI_ST_SINGULAR, n = 169 TWXI_ST_LIMIT, failed points NaN.  Bitwise: mth = 0 equals every
    mth = m call, a repeated call is identical, and krig_all's vario equals fit_vario at the same counts."""
    stats, bad = _Stats(), []
    for v in dense:
        for z in (False, True):
            sel = np.flatnonzero(v["rmz"] == z)
            vario, st = _fit_batch(v, sel, COUNTS)
            vario2, st2 = _fit_batch(v, sel, COUNTS)
            assert np.array_equal(vario, vario2, equal_nan=True) and np.array_equal(st, st2)
            for m in (1, 5, 12):
                vm, stm = _fit_batch(v, sel, COUNTS, mth=m)
                assert np.array_equal(vm[:, 0], vario[:, m - 1], equal_nan=True) and np.array_equal(stm, st), m
            for r in range(st.size):
                q, n = sel[r // len(COUNTS)], COUNTS[r % len(COUNTS)]
                for m in (range(1, 13) if n <= 65 else BIG_MONTHS):
                    _compare(stats, bad, "dense", (v["w"], q, n, m), vario[r, m - 1], st[r], v["ref"][q, n, m])
            # krig_all: variogram fit and kriging in one call; its vario is the same kernel at the same counts
            nc = len(COUNTS)
            lat, lon = np.repeat(v["lat"][sel], nc), np.repeat(v["lon"][sel], nc)
            elev = v["f"].elev(lon, lat)
            lst = np.stack([v["f"].lst(v["w"], m, lon, lat, elev) for m in range(1, 13)], axis=1)
            nn = np.tile(np.asarray(COUNTS, dtype=np.int32), len(sel))
            _, _, kv, kst = v["ctx"].krig_all(lat, lon, elev, lst, nn, rm_zero=z)
            ok = kst == ST_OK
            assert np.array_equal(kv[ok], vario[ok]) and np.all(st[~ok] != ST_OK)
    stats.report("vario_fit_kernel, dense table, against vario_exact")
    assert not bad, (len(bad), bad[:6])


@pytest.mark.gpu
def test_fit_vario_alone_equals_in_shuffled_batch(dense):
    """A point fitted alone gives the bits it gets inside a shuffled batch of 2400 points (fixed-point lag sums and a
    fixed reduction order: nothing depends on the batch or on atomics' timing)."""
    v = dense[1]
    rng = np.random.default_rng(3)
    lat = rng.uniform(v["lat"].min(), v["lat"].max(), 2400)
    lon = rng.uniform(v["lon"].min(), v["lon"].max(), 2400)
    nn = rng.choice([7, 16, 33, 64, 128, 168], 2400).astype(np.int32)
    vb, sb = v["ctx"].fit_vario(lat, lon, nnghs=nn)
    for i in rng.choice(2400, 12, replace=False):
        va, sa = v["ctx"].fit_vario(lat[i:i + 1], lon[i:i + 1], nnghs=nn[i:i + 1])
        assert sa[0] == sb[i] and np.array_equal(va[0], vb[i], equal_nan=True), i


# ---- 2. sparse table: hundreds of lags, both sides of the 512-lag limit ---------------------------------------------
@pytest.mark.gpu
def test_fit_vario_sparse_lags_vs_exact():
    """A few hundred stations over CONUS: at n up to 168 the cutoff spans hundreds of 5 km lags.  Points whose lag
    count nb = floor(1.4 dist[n-1] / 5) + 1 is just below 512 are fitted, those just above are TWXI_ST_LIMIT."""
    from topowx_b200 import synth, db
    from topowx_b200.context import TwxiContext
    f = synth.Fields()
    d = synth.make_station_db(1, 400, synth.conus_bbox(), f, synth.make_days(1995, 1))
    ctx = TwxiContext(d, np.isnan(d.stns[db.BAD]))
    rng = np.random.default_rng(11)
    lat = rng.uniform(30.0, 46.0, 64)
    lon = rng.uniform(-118.0, -75.0, 64)
    idx, dist, _, st = ctx.knn(lat, lon, MAX_N)
    assert np.all(st == 0)
    gidx = ctx.gidx[idx]
    nb = np.floor(dist[:, :MAX_N] * 1.4 / WIDTH).astype(np.int64) + 1
    cm = []
    below = above = 0
    for q in range(lat.size):
        under = np.flatnonzero((nb[q] <= MAXBIN) & (np.arange(1, MAX_N + 1) >= 7))
        over = np.flatnonzero(nb[q] > MAXBIN)
        if under.size:
            cm.append((q, int(under[-1]) + 1, 1 + q % 12))                  # the largest count within the limit
            cm.append((q, int(under[under.size // 2]) + 1, 1 + (q + 5) % 12))
        if over.size:
            cm.append((q, int(over[0]) + 1, 1 + (q + 3) % 12))              # the smallest count beyond it
    tasks, meta = _tasks(d, gidx, dist, cm)
    refs = _farm(tasks)
    stats, bad = _Stats(), []
    nbs = []
    for (q, n, m), ref in zip(meta, refs):
        vario, st = ctx.fit_vario(lat[q:q + 1], lon[q:q + 1], mth=m, nnghs=np.array([n], dtype=np.int32))
        _compare(stats, bad, "sparse", (q, n, m), vario[0, 0], st[0], ref)
        if ref["status"] == ST_LIMIT:
            above += 1
        elif ref["status"] == ST_OK:
            nbs.append(ref["nb"])
            below += ref["nb"] >= MAXBIN - 40
    stats.report("vario_fit_kernel, sparse table, against vario_exact (nb up to %d)" % max(nbs))
    assert below >= 3 and above >= 3, (below, above)
    assert not bad, (len(bad), bad[:6])


# ---- 3. constructed neighbourhoods -----------------------------------------------------------------------------------
def _edited(d, stns):
    from topowx_b200 import db
    from topowx_b200.context import TwxiContext
    e = db.StationSerialDataDb((stns, d.var, d.days), d.var_name)
    return e, TwxiContext(e, np.isnan(stns[db.BAD]))


@pytest.mark.gpu
def test_fit_vario_constructed_cases(dense):
    """Edited copies of the dense table: (a) normals scaled by 2^-6 and 2^6 (nugget and psill scale by 4^-6 / 4^6 in the
    reference, the range stays; at 2^-6 the fixed-point floor of the lag sums is 4096 times closer to gamma); (b) a tight
    cluster of 9 stations whose pairs all fall into lag 0 (K = 1); (c) two stations moved onto one location: every point
    that sees both is TWXI_ST_SINGULAR (decided exactly, also for a pure nugget), the others keep their bits."""
    from topowx_b200 import db
    v = dense[0]
    d = v["d"]
    stats, bad = _Stats(), []
    lat, lon = v["lat"][:6], v["lon"][:6]
    counts = [7, 16, 33, 64]
    base, bst = v["ctx"].fit_vario(np.repeat(lat, 4), np.repeat(lon, 4), nnghs=np.tile(np.int32(counts), 6))
    # (a) scaled normals
    for sc in (2.0 ** -6, 2.0 ** 6):
        s = d.stns.copy()
        for m in range(1, 13):
            s[db.get_norm_varname(m)] = s[db.get_norm_varname(m)] * sc
        e, ctx = _edited(d, s)
        vario, st = ctx.fit_vario(np.repeat(lat, 4), np.repeat(lon, 4), nnghs=np.tile(np.int32(counts), 6))
        assert np.array_equal(st, bst)
        cm = [(q, n, m) for q in range(6) for n in counts for m in (2, 8)]
        tasks, meta = _tasks(e, v["gidx"], v["dist"], cm)
        for (q, n, m), ref in zip(meta, _farm(tasks)):
            r0 = v["ref"][q, n, m]
            if r0["status"] == ST_OK and ref["status"] == ST_OK:
                # the reference itself: exact scaling (powers of two), to its 40-digit rounding
                np.testing.assert_allclose(ref["out"], r0["out"] * np.array([sc * sc, sc * sc, 1.0]), rtol=1e-25)
            _compare(stats, bad, "scaled %g" % sc, (q, n, m), vario[q * 4 + counts.index(n), m - 1], st[q * 4 + counts.index(n)],
                     ref)
    # (b) K = 1: the 9 nearest stations of cell 0 moved into a 2 km cluster around it (pairs < 5 km)
    s = d.stns.copy()
    near = v["gidx"][0, :9]
    ang = np.linspace(0.0, 2 * np.pi, 9, endpoint=False)
    s[db.LAT][near] = lat[0] + 0.008 * np.sin(ang) * (1 + 0.1 * np.arange(9))
    s[db.LON][near] = lon[0] + 0.010 * np.cos(ang) * (1 + 0.1 * np.arange(9))
    e, ctx = _edited(d, s)
    idx, dist, _, _ = ctx.knn(lat[:1], lon[:1], 9)
    gidx = ctx.gidx[idx]
    assert set(gidx[0, :9]) == set(near)
    vario, st = ctx.fit_vario(lat[:1], lon[:1], nnghs=np.array([9], dtype=np.int32))
    tasks, meta = _tasks(e, gidx, dist, [(0, 9, m) for m in range(1, 13)])
    nk1 = 0
    for (q, n, m), ref in zip(meta, _farm(tasks)):
        nk1 += ref.get("K") == 1
        _compare(stats, bad, "cluster", (q, n, m), vario[0, m - 1], st[0], ref)
    assert nk1 == 12
    # (c) a co-located pair: the 2 nearest stations of cell 0
    s = d.stns.copy()
    a, b = v["gidx"][0, :2]
    s[db.LON][b], s[db.LAT][b] = s[db.LON][a], s[db.LAT][a]
    e, ctx = _edited(d, s)
    nn = np.tile(np.int32(counts), 6)
    vario, st = ctx.fit_vario(np.repeat(lat, 4), np.repeat(lon, 4), nnghs=nn)
    idx, _, _, _ = ctx.knn(np.repeat(lat, 4), np.repeat(lon, 4), max(counts))
    gi = ctx.gidx[idx]
    idx0, _, _, _ = v["ctx"].knn(np.repeat(lat, 4), np.repeat(lon, 4), max(counts))
    gi0 = v["ctx"].gidx[idx0]
    nsing = 0
    for r in range(nn.size):
        sees = a in gi[r, :nn[r]] and b in gi[r, :nn[r]]
        if sees:
            nsing += 1
            assert st[r] == ST_SINGULAR and np.all(np.isnan(vario[r])), r
            with pytest.raises(o.OracleError) as ex:
                sel = gi[r, :nn[r]]
                o.get_vario_params(s[db.LON][sel], s[db.LAT][sel], np.column_stack(_arrays(e, sel, 1)[:4]),
                                   s[db.get_norm_varname(1)][sel], np.ones(sel.size))
            assert ex.value.status == o.ST_SINGULAR
        elif b not in gi[r, :nn[r]] and np.array_equal(gi[r, :nn[r]], gi0[r, :nn[r]]):
            assert st[r] == bst[r] and np.array_equal(vario[r], base[r], equal_nan=True), r
    assert nsing >= 4
    stats.report("vario_fit_kernel, constructed neighbourhoods, against vario_exact")
    assert not bad, (len(bad), bad[:6])


# ---- 4. the reference itself (CPU) ----------------------------------------------------------------------------------
def _neighbourhood(rng, n):
    lon = rng.uniform(-100, -97, n)
    lat = rng.uniform(38, 41, n)
    elev = rng.uniform(200, 2500, n)
    lst = 30.0 - 0.006 * elev + rng.normal(0, 0.4, n)
    H = o.gcdist_sp(lon[:, None], lat[:, None], lon[None, :], lat[None, :])
    L = np.linalg.cholesky(np.exp(-H / rng.uniform(30, 300)) + 1e-9 * np.eye(n))
    y = 20.0 - 0.0065 * elev + 0.2 * lst + L @ rng.normal(size=n) * 0.7 + rng.normal(size=n) * rng.uniform(0.05, 0.5)
    far = o.gcdist_sp(-98.5, 39.5, lon, lat)
    order = np.argsort(far)
    return lon[order], lat[order], elev[order], lst[order], y[order], float(far[order][-1])


def test_exact_reference_vs_oracle_and_stationary():
    """On random neighbourhoods vario_exact agrees with the (polished) float64 oracle within its bound, and its range
    is a stationary point of S: |S'(r*)| r* <= 1e-28 S with S'' > 0."""
    rng = np.random.default_rng(5)
    nchk = 0
    for n in (7, 12, 30, 60, 90):
        lon, lat, elev, lst, y, dmax = _neighbourhood(rng, n)
        ref = vario_exact(lon, lat, elev, lst, y, dmax)
        assert ref["status"] == ST_OK
        X = np.column_stack([lon, lat, elev, lst])
        ov = np.array(o.get_vario_params(lon, lat, X, y, np.full(n, dmax)))
        if ref["branch2"] == "range":
            assert abs(ref["g2"]) * ref["out"][2] <= 1e-28 * ref["S2"] and ref["gp2"] < 0
        if ref["near"] or not ref["stage5_comparable"] or (ref["branch2"] == "range" and not ref["ident"]):
            continue
        nchk += 1
        assert np.all(np.abs(ov - ref["out"]) <= ref["bound"]), (n, ov, ref["out"], ref["bound"])
    assert nchk >= 3


def test_oracle_range_fit_reaches_exact_root():
    """oracle.fit_exp_range (the algorithm of vario.cu's fit_range_warp, with its Newton polish) lands within 1e-14
    relative of the 40-digit root of dS/dr on 100 random neighbourhoods; flat (non-identifiable) ones are counted."""
    rng = np.random.default_rng(1)
    errs, flat = [], 0
    while len(errs) < 100:
        n = int(rng.integers(20, 150))
        lon, lat, elev, lst, y, dmax = _neighbourhood(rng, n)
        H = o.gcdist_sp(lon[:, None], lat[:, None], lon[None, :], lat[None, :])
        z = y - y.mean()
        npairs, dist, gamma = o.sample_variogram(H, z, dmax * 0.7)
        sill, nug = float(np.var(z, ddof=1)), float(np.min(gamma))
        m = o.fit_exp_range(npairs, dist, gamma, nug, sill)
        with mpmath.workdps(DPS):
            f = _fit(list(npairs), [_mp(t) for t in dist], [_mp(t) for t in gamma], _mp(sill))
        if m is None or f["branch"] != "range":
            assert m is None or f["branch"] in ("range", "noroot")
            continue
        if not f["ident"]:
            flat += 1
            continue
        errs.append(abs(m[2] - float(f["r"])) / float(f["r"]))
    print("\noracle range vs 40-digit root: median %.3g, max %.3g relative (%d flat skipped)"
          % (np.median(errs), np.max(errs), flat))
    assert max(errs) <= 1e-14


def test_colocated_and_fewer_than_7_are_singular():
    """Co-located neighbours and n < 7 raise OracleError(ST_SINGULAR) in the oracle and give ST_SINGULAR in the
    reference, every time."""
    rng = np.random.default_rng(9)
    for n in (6, 7, 20, 60):
        lon, lat, elev, lst, y, dmax = _neighbourhood(rng, n)
        for trial in range(2 if n >= 7 else 1):
            if n >= 7:
                i, j = rng.choice(n, 2, replace=False)
                lon[j], lat[j] = lon[i], lat[i]
            X = np.column_stack([lon, lat, elev, lst])
            with pytest.raises(o.OracleError) as e:
                o.get_vario_params(lon, lat, X, y, np.full(n, dmax))
            assert e.value.status == o.ST_SINGULAR
            assert vario_exact(lon, lat, elev, lst, y, dmax)["status"] == ST_SINGULAR
    for n in range(1, 7):
        lon, lat, elev, lst, y, dmax = _neighbourhood(rng, 7)
        with pytest.raises(o.OracleError):
            o.get_vario_params(lon[:n], lat[:n], np.column_stack([lon, lat, elev, lst])[:n], y[:n], np.full(n, dmax))

"""numpy FP64 restatement of the TopoWx interpolation hot path (CPU oracle).

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``): imported by ``tests/``, ``smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py``; never by ``topowx_b200``.

Every function cites the reference lines it follows (paths under ``/root/reference``).  The module is
standalone: it needs numpy only and never reads the reference tree, so it travels to the GPU box.

Inputs are plain containers:
  * ``stns``  – numpy structured array with the reference's field names
                (``twx/db/station_data.py:49-124``): station_id, longitude, latitude, elevation, tdi,
                mask, bad, climdiv, normMM, lstMM, optim_nnghsMM, optim_nnghs_animMM,
                vario_nugMM / vario_psillMM / vario_rngMM (MM = 01..12); numeric fields float64.
  * ``obs``   – float32 [ndays, N] in DB (= station-id) order, no missing values.
  * ``days``  – structured array with YEAR / MONTH fields (``twx/utils/util_dates.py:150-159``).

Kriging: ``ked_gstat`` restates what R ``gstat::krige`` does for ``krig_meantair``
(``twx/interp/rpy/interp.R:198-270``) – PARITY UNPINNED against real gstat (not installable here);
pinned by analytic known answers in ``tests/test_oracle_ked.py``.
"""
import numpy as np

# field names: twx/db/station_data.py:49-68
LON, LAT, ELEV, TDI, LST = "longitude", "latitude", "elevation", "tdi", "lst"
STN_ID, MASK, BAD, CLIMDIV = "station_id", "mask", "bad", "climdiv"
YEAR, MONTH = "YEAR", "MONTH"
KRIG_TREND_VARS = (LON, LAT, ELEV, LST)            # interp_tair.py:46
GWR_TREND_VARS = (LON, LAT, ELEV, TDI, LST)        # interp_tair.py:47
KED_MIN_NNGHS = 1 + len(KRIG_TREND_VARS)           # fewer neighbours: the kriging trend matrix is singular
DFLT_INIT_NNGHS = 100                              # interp_tair.py:51
RADIAN_CONVERSION_FACTOR = 0.017453292519943295    # util_geo.py:21
AVG_EARTH_RADIUS_KM = 6371.009                     # util_geo.py:22
FILL_I2, FILL_I4 = -32767, -2147483647             # netCDF4.default_fillvals (step25:73-88)
FILL_F4 = np.float32(9.969209968386869e+36)
SCALE_FACTOR = np.float32(0.01)                    # step25:45

# per-cell status codes shared with include/twxi.h (SURVEY §8b error conventions)
ST_OK, ST_NO_NNGHS, ST_NO_VARIO, ST_TOO_FEW_STNS, ST_SINGULAR, ST_FIXER_EMPTY, ST_CLIMDIV = range(7)


def lst_name(m):   return "lst%02d" % m              # station_data.py:104-109
def norm_name(m):  return "norm%02d" % m             # station_data.py:111-116
def optim_name(m): return "optim_nnghs%02d" % m      # station_data.py:118-123
def optim_anom_name(m): return "optim_nnghs_anom%02d" % m   # station_data.py:125-130
def vario_name(m, p): return "%s%02d" % (p, m)       # station_data.py:132-138


class OracleError(Exception):
    """Per-point failure; ``status`` is the code the C ABI reports for the same condition."""

    def __init__(self, status, msg):
        Exception.__init__(self, msg)
        self.status = status


# ------------------------------------------------------------------------------------------------
# a1  twx/utils/util_geo.py:24-40
def grt_circle_dist(lon1, lat1, lon2, lat2):
    lat1rad = lat1 * RADIAN_CONVERSION_FACTOR
    lat2rad = lat2 * RADIAN_CONVERSION_FACTOR
    lon1rad = lon1 * RADIAN_CONVERSION_FACTOR
    lon2rad = lon2 * RADIAN_CONVERSION_FACTOR
    deltaLat = lat1rad - lat2rad
    deltaLon = lon1rad - lon2rad
    centralangle = 2 * np.arcsin(np.sqrt((np.sin(deltaLat / 2)) ** 2
                                         + np.cos(lat1rad) * np.cos(lat2rad) * (np.sin(deltaLon / 2)) ** 2))
    return AVG_EARTH_RADIUS_KM * centralangle


class StationDb(object):
    """Minimal stand-in for ``StationSerialDataDb`` (station_data.py:547-666) over in-memory arrays."""

    def __init__(self, stns, obs, days):
        self.stns = stns
        self.stn_ids = stns[STN_ID]
        self.obs = obs
        self.days = days
        self.mth_idx = {m: np.nonzero(days[MONTH] == m)[0] for m in range(1, 13)}   # :576-580
        self.mth_idx[None] = np.arange(days.size)
        self.stn_idxs = {sid: i for i, sid in enumerate(self.stn_ids)}              # :608-610

    def load_obs(self, stn_ids, mth=None):
        # station_data.py:619-666 / interp_tair.py:1084-1095: columns come back in DB order
        mask = np.nonzero(np.isin(self.stn_ids, stn_ids))[0]
        obs = self.obs[:, mask]
        if mth is not None:
            obs = np.take(obs, self.mth_idx[mth], axis=0)
        return obs


# ------------------------------------------------------------------------------------------------
# a2/a3  twx/interp/station_select.py
class StationSelect(object):
    """station_select.py:29-192.  The only deliberate difference: ``argsort(kind='stable')`` instead
    of the default unstable sort (:111), i.e. the north_star tie-break (distance, then station index)."""

    def __init__(self, stn_da, stn_mask=None, rm_zero_dist_stns=False):
        self.stn_da = stn_da
        if stn_mask is None:                                   # :52-55
            self.stns = stn_da.stns
            self.stn_gidx = np.arange(stn_da.stns.size)
        else:
            self.stns = stn_da.stns[stn_mask]
            self.stn_gidx = np.nonzero(stn_mask)[0]
        self.rm_zero_dist_stns = rm_zero_dist_stns
        self._key = None

    def _set_pt(self, lat, lon, stns_rm=None):                 # :72-119
        if isinstance(stns_rm, str):
            stns_rm = np.array([stns_rm])
        key = (lat, lon, None if stns_rm is None else tuple(stns_rm))
        if key == self._key:                                   # cache :79-91
            return
        stn_dists = grt_circle_dist(lon, lat, self.stns[LON], self.stns[LAT])       # :93
        fnl_rm = stns_rm if stns_rm is not None else np.array([], dtype=self.stns[STN_ID].dtype)
        if self.rm_zero_dist_stns:                             # :97-99
            fnl_rm = np.unique(np.concatenate((fnl_rm, self.stns[STN_ID][stn_dists == 0])))
        if fnl_rm.size > 0:                                    # :101-104
            mask_rm = np.logical_not(np.isin(self.stns[STN_ID], fnl_rm))
        else:
            mask_rm = np.ones(self.stns.size, dtype=bool)
        order = np.argsort(stn_dists, kind="stable")           # :111 (stable = spec'd tie-break)
        order = order[mask_rm[order]]                          # :115-119
        self.pt_sort_idx = order                               # index into self.stns
        self.pt_sort_stn_dists = stn_dists[order]
        self._key = key

    def set_ngh_stns(self, lat, lon, nnghs, load_obs=True, obs_mth=None, stns_rm=None):   # :121-192
        self._set_pt(lat, lon, stns_rm)
        d = self.pt_sort_stn_dists
        if nnghs >= d.size:                                    # IndexError at :164
            raise OracleError(ST_TOO_FEW_STNS, "index %d is out of bounds" % nnghs)
        dbw = d[nnghs]                                         # :164
        idx = self.pt_sort_idx[0:nnghs]
        dists = d[0:nnghs]
        wgt = np.square(1.0 - np.square(dists / dbw))          # :169
        # :179-182 sort by station id.  DB order is station-id order (create_db_all_stations.py:509-515)
        # so sorting the row index is the same permutation as sorting the id strings.
        stnid_sort = np.argsort(self.stns[STN_ID][idx], kind="stable")
        self.ngh_idx_dist_order = idx
        self.ngh_idx = idx[stnid_sort]
        self.ngh_stns = self.stns[self.ngh_idx]
        self.ngh_wgt = wgt[stnid_sort]
        self.ngh_dists = dists[stnid_sort]
        if load_obs:                                           # :184-187
            self.ngh_obs = self.stn_da.load_obs(self.stns[STN_ID][idx], mth=obs_mth)
        else:
            self.ngh_obs = None


# ------------------------------------------------------------------------------------------------
# a7  R krig_meantair -> gstat::krige (interp.R:198-270)   [EXT: gstat 1.0-25 / sp 1.1-1]
def gcdist_sp(lon1, lat1, lon2, lat2):
    """WGS-84 great-circle distance (km) as in sp's ``sp_gcdist`` C routine, which gstat copies for
    unprojected (+proj=longlat) data (interp.R:218-221): Andoyer-Lambert / Meeus form, a = 6378.137 km,
    f = 1/298.257223563; identical points (|dlat|,|dlon| < DBL_EPSILON) -> 0.  Vectorised over arrays."""
    lon1, lat1, lon2, lat2 = np.broadcast_arrays(np.asarray(lon1, dtype=np.float64), np.asarray(lat1, dtype=np.float64),
                                                 np.asarray(lon2, dtype=np.float64), np.asarray(lat2, dtype=np.float64))
    DE2RA = np.pi / 180.0
    a = 6378.137
    f = 1.0 / 298.257223563
    eps = np.finfo(np.float64).eps
    same = (np.abs(lat1 - lat2) < eps) & ((np.abs(lon1 - lon2) < eps) |
                                          (np.abs((np.abs(lon1) + np.abs(lon2)) - 360.0) < eps))
    lat1R, lat2R, lon1R, lon2R = lat1 * DE2RA, lat2 * DE2RA, lon1 * DE2RA, lon2 * DE2RA
    F = (lat1R + lat2R) / 2.0
    G = (lat1R - lat2R) / 2.0
    L = (lon1R - lon2R) / 2.0
    sinG2, cosG2 = np.sin(G) ** 2, np.cos(G) ** 2
    sinF2, cosF2 = np.sin(F) ** 2, np.cos(F) ** 2
    sinL2, cosL2 = np.sin(L) ** 2, np.cos(L) ** 2
    S = sinG2 * cosL2 + cosF2 * sinL2
    C = cosG2 * cosL2 + sinF2 * sinL2
    with np.errstate(all="ignore"):
        w = np.arctan(np.sqrt(S / C))
        R = np.sqrt(S * C) / w
        D = 2 * w * a
        H1 = (3 * R - 1) / (2 * C)
        H2 = (3 * R + 1) / (2 * S)
        d = D * (1 + f * H1 * sinF2 * cosG2 - f * H2 * cosF2 * sinG2)
    return np.where(same, 0.0, d)


def covariance_gstat(h, nug, psill, rng):
    """gstat covariance for ``vgm(model='Exp', nugget, psill, range)`` – C(h) = psill*exp(-h/range) for
    h > 0 and nug + psill at h == 0 – or for the pure nugget ``vgm(psill+nug, 'Nug')`` used when
    range == 0 (interp.R:223-231)."""
    h = np.asarray(h, dtype=np.float64)
    if rng == 0:
        return np.where(h == 0, nug + psill, 0.0)
    return np.where(h == 0, nug + psill, psill * np.exp(-h / rng))


def ked_gstat(ngh_lon, ngh_lat, ngh_X, ngh_y, pt_lon, pt_lat, pt_x, nug, psill, rng):
    """Kriging with external drift at one point, all n neighbours used (no nmax) – what
    ``krige(tair~longitude+latitude+elevation+lst, stns_ngh, newdata=pt, model)`` computes
    (interp.R:256-258).  ``ngh_X`` is n x 4 (lon, lat, elev, lst); intercept is added here.

    mean = x0'b + c0'V^-1(y - Xb),  b = (X'V^-1X)^-1 X'V^-1 y
    var  = C(0) - c0'V^-1c0 + (x0 - X'V^-1c0)'(X'V^-1X)^-1(x0 - X'V^-1c0)

    The drift columns are centred on the prediction point and scaled before factorising; with an
    intercept in X this is an exact reparametrisation of the same predictor (tests compare it with
    the uncentred augmented system solved in extended precision).
    Raises OracleError(ST_SINGULAR) where R would stop with a singular covariance matrix, and for fewer than 5
    neighbours: X'V^-1X of the intercept and four drift columns is then singular in exact arithmetic, whatever the
    rounded Cholesky factorisation of it says."""
    n = ngh_lon.size
    if n < KED_MIN_NNGHS:
        raise OracleError(ST_SINGULAR, "fewer than 5 neighbours: singular trend matrix")
    H = gcdist_sp(ngh_lon[:, None], ngh_lat[:, None], ngh_lon[None, :], ngh_lat[None, :])
    V = covariance_gstat(H, nug, psill, rng)
    V[np.diag_indices(n)] = nug + psill
    c0 = covariance_gstat(gcdist_sp(pt_lon, pt_lat, ngh_lon, ngh_lat), nug, psill, rng)
    Xc = np.asarray(ngh_X, dtype=np.float64) - np.asarray(pt_x, dtype=np.float64)[None, :]
    scale = np.max(np.abs(Xc), axis=0)
    scale[scale == 0] = 1.0
    X = np.column_stack((np.ones(n), Xc / scale))
    x0 = np.zeros(X.shape[1])
    x0[0] = 1.0
    yref = ngh_y[0]
    y = ngh_y - yref
    try:
        Lc = np.linalg.cholesky(V)
    except np.linalg.LinAlgError:
        raise OracleError(ST_SINGULAR, "singular covariance matrix")
    from numpy.linalg import solve
    B = solve(Lc, np.column_stack((X, y, c0)))          # L^-1 [X | y | c0]
    A, b, c = B[:, :-2], B[:, -2], B[:, -1]
    G = A.T @ A
    try:
        Lg = np.linalg.cholesky(G)
    except np.linalg.LinAlgError:
        raise OracleError(ST_SINGULAR, "singular trend matrix")
    r = x0 - A.T @ c
    t = solve(Lg.T, solve(Lg, r))
    mean = t @ (A.T @ b) + c @ b + yref
    var = (nug + psill) - c @ c + r @ t
    if not (np.isfinite(mean) and np.isfinite(var)):
        raise OracleError(ST_SINGULAR, "non-finite kriging result")
    return float(mean), float(var)


# ------------------------------------------------------------------------------------------------
# a9  interp_tair.py:1099-1146
def gwr_series(model_x, predict_x, y, wgt):
    model_x = np.require(model_x, dtype=np.float64)
    predict_x = np.require(predict_x, dtype=np.float64)
    y = np.require(y, dtype=np.float64)
    wgt = np.require(wgt, dtype=np.float64)
    X = np.column_stack((np.ones(model_x.shape[0]), model_x))      # :1128
    x = np.insert(predict_x, 0, 1)                                 # :1129
    x.shape = (x.shape[0], 1)
    XtW = X.T * wgt[None, :]                                       # == dot(X_t, diag(w))  :1132-1137
    m1 = np.linalg.inv(np.dot(XtW, X))                             # :1136
    m3 = np.dot(m1, XtW)                                           # :1138
    z = np.dot(np.transpose(x), m3)                                # :1140
    return np.inner(z, y).ravel(), z.ravel()                       # :1143


# ------------------------------------------------------------------------------------------------
# a4-a6, a8, a10
class KrigTair(object):
    """interp_tair.py:770-926 with the R call replaced by :func:`ked_gstat`."""

    def __init__(self, stn_slct):
        self.stn_slct = stn_slct

    def std_err_ci(self, tair_mean, tair_var):                     # :794-819
        std_err = np.sqrt(tair_var) if tair_var >= 0 else 0
        ci_r = np.abs(std_err * -1.959963984540054)                # stats.norm.ppf(0.025) :792
        return std_err, (tair_mean - ci_r, tair_mean + ci_r)

    def get_nnghs(self, pt, mth, stns_rm=None):                    # :821-835
        ss = self.stn_slct
        ss.set_ngh_stns(pt[LAT], pt[LON], DFLT_INIT_NNGHS, load_obs=False, stns_rm=stns_rm)
        fin = np.isfinite(ss.ngh_stns[optim_name(mth)])
        if fin.sum() == 0:
            raise OracleError(ST_NO_NNGHS, "Cannot determine the optimal # of neighbors to use!")
        return int(np.round(np.average(ss.ngh_stns[optim_name(mth)][fin], weights=ss.ngh_wgt[fin])))

    def get_vario_params(self, pt, mth):                           # :837-851
        ss = self.stn_slct
        fin = np.isfinite(ss.ngh_stns[vario_name(mth, "vario_nug")])
        if fin.sum() == 0:
            raise OracleError(ST_NO_VARIO, "Cannot determine variogram params!")
        w = ss.ngh_wgt[fin]
        s = ss.ngh_stns[fin]
        return (np.average(s[vario_name(mth, "vario_nug")], weights=w),
                np.average(s[vario_name(mth, "vario_psill")], weights=w),
                np.average(s[vario_name(mth, "vario_rng")], weights=w))

    def krig(self, pt, mth, nnghs=None, vario_params=None, stns_rm=None):   # :853-926
        ss = self.stn_slct
        if nnghs is None:
            nnghs = self.get_nnghs(pt, mth, stns_rm)
        ss.set_ngh_stns(pt[LAT], pt[LON], nnghs, load_obs=False, stns_rm=stns_rm)
        nug, psill, vrange = self.get_vario_params(pt, mth) if vario_params is None else vario_params
        nghs = ss.ngh_stns
        X = np.column_stack([nghs[LON], nghs[LAT], nghs[ELEV], nghs[lst_name(mth)]])
        x = np.array([pt[LON], pt[LAT], pt[ELEV], pt[lst_name(mth)]], dtype=np.float64)
        self.last = dict(nnghs=nnghs, nug=nug, psill=psill, rng=vrange, idx=ss.ngh_idx_dist_order.copy())
        return ked_gstat(nghs[LON], nghs[LAT], X, nghs[norm_name(mth)], pt[LON], pt[LAT], x, nug, psill, vrange)


class GwrTairAnom(object):
    """interp_tair.py:215-314."""

    def __init__(self, stn_slct):
        self.stn_slct = stn_slct

    def get_nnghs(self, pt, mth, stns_rm=None):                    # :245-259
        ss = self.stn_slct
        ss.set_ngh_stns(pt[LAT], pt[LON], DFLT_INIT_NNGHS, load_obs=False, stns_rm=stns_rm)
        fin = np.isfinite(ss.ngh_stns[optim_anom_name(mth)])
        if fin.sum() == 0:
            raise OracleError(ST_NO_NNGHS, "Cannot determine the optimal # of neighbors to use!")
        return int(np.round(np.average(ss.ngh_stns[optim_anom_name(mth)][fin], weights=ss.ngh_wgt[fin])))

    def gwr_mth(self, pt, mth, nnghs=None, stns_rm=None):          # :261-314
        ss = self.stn_slct
        if nnghs is None:
            nnghs = self.get_nnghs(pt, mth, stns_rm)
        ss.set_ngh_stns(pt[LAT], pt[LON], nnghs, load_obs=True, stns_rm=stns_rm, obs_mth=mth)
        ngh_obs_cntr = ss.ngh_obs - ss.ngh_stns[norm_name(mth)]   # :300  (f4 - f8 -> f8)
        preds = [v if v != LST else lst_name(mth) for v in GWR_TREND_VARS]
        X = np.column_stack([ss.ngh_stns[v] for v in preds])       # :303-304
        x = np.array([pt[v] for v in preds], dtype=np.float64)     # :306-307
        interp_anom, z = gwr_series(X, x, ngh_obs_cntr, ss.ngh_wgt)    # :309
        self.last = dict(nnghs=nnghs, z=z, idx=ss.ngh_idx.copy())
        return interp_anom + pt[norm_name(mth)]                    # :312


class InterpTair(object):
    """interp_tair.py:371-439."""

    def __init__(self, krig_tair, gwr_tair):
        self.krig_tair = krig_tair
        self.gwr_tair = gwr_tair
        self.mth_masks = gwr_tair.stn_slct.stn_da.mth_idx
        self.ndays = gwr_tair.stn_slct.stn_da.days.size

    def interp(self, pt, stns_rm=None, norms_only=False):          # :396-439
        tair_daily = np.zeros(self.ndays)
        tair_norms = np.zeros(12)
        tair_se = np.zeros(12)
        self.tair_var = np.zeros(12)
        for mth in range(1, 13):
            tair_mean, tair_var = self.krig_tair.krig(pt, mth, stns_rm=stns_rm)
            std_err, _ = self.krig_tair.std_err_ci(tair_mean, tair_var)
            pt[norm_name(mth)] = tair_mean
            tair_norms[mth - 1] = tair_mean
            tair_se[mth - 1] = std_err
            self.tair_var[mth - 1] = tair_var
            if not norms_only:
                tair_daily[self.mth_masks[mth]] = self.gwr_tair.gwr_mth(pt, mth, stns_rm=stns_rm)
        return tair_daily, tair_norms, tair_se


# a12  interp_tair.py:143-197
def tmin_tmax_fixer(tmin, tmax, tail=15):
    invalid_days = np.nonzero(tmin >= tmax)[0]
    if invalid_days.size > 0:
        tmin = np.copy(tmin)
        tmax = np.copy(tmax)
        for x in invalid_days:
            tavg = (tmin[x] + tmax[x]) / 2.0
            start = max(x - tail, 0)
            end = min(x + tail + 1, tmin.size)
            tmin_win = tmin[start:end]
            tmax_win = tmax[start:end]
            mask = tmin_win < tmax_win
            if mask.sum() == 0:
                raise OracleError(ST_FIXER_EMPTY, "No valid tmin/tmax in window")
            tdir_half = np.mean(tmax_win[mask] - tmin_win[mask], dtype=np.float64) / 2.0
            tmin[x] = tavg - tdir_half
            tmax[x] = tavg + tdir_half
    return tmin, tmax, invalid_days.size


def build_empty_pt():                                              # interp_tair.py:200-213
    dt = [(LON, np.float64), (LAT, np.float64), (ELEV, np.float64), (TDI, np.float64),
          (CLIMDIV, np.float64), (MASK, np.float64)]
    dt += [("tmin%02d" % m, np.float64) for m in range(1, 13)]
    dt += [("tmax%02d" % m, np.float64) for m in range(1, 13)]
    dt += [(norm_name(m), np.float64) for m in range(1, 13)]
    dt += [(optim_name(m), np.float64) for m in range(1, 13)]
    dt += [(lst_name(m), np.float64) for m in range(1, 13)]
    dt += [(optim_anom_name(m), np.float64) for m in range(1, 13)]
    return np.zeros(1, dtype=dt)[0]


def _rgn_nnghs_keys(stns):                                         # interp_tair.py:594-610 (keys only)
    c = stns[CLIMDIV]
    return set(np.unique(c[np.isfinite(c)]).tolist())


class PtInterpTair(object):
    """interp_tair.py:441-592 (aux_fpaths / interp_to_lonlat are raster I/O, out of scope)."""

    def __init__(self, stn_da_tmin, stn_da_tmax):
        self.days = stn_da_tmin.days
        days = self.days
        self.daysNormMask = np.nonzero((days[YEAR] >= 1981) & (days[YEAR] <= 2010))[0]    # :466
        daysNorm = days[self.daysNormMask]
        uYrs = np.unique(daysNorm[YEAR])
        if uYrs.size == 0:
            raise IndexError("no days within 1981-2010")           # uYrs[0] at :470
        self.yrMthsMasks = [np.nonzero((daysNorm[YEAR] == y) & (daysNorm[MONTH] == m))[0]
                            for y in uYrs for m in range(1, 13)]   # :472-475
        # get_mth_metadata(uYrs[0], uYrs[-1]) covers every year in the range (:470, :477-479)
        yr_mths_month = np.tile(np.arange(1, 13), int(uYrs[-1] - uYrs[0] + 1))
        self.mth_masks = [np.nonzero(yr_mths_month == m)[0] for m in range(1, 13)]
        mask_tmin = np.isnan(stn_da_tmin.stns[BAD])                # :481-482
        mask_tmax = np.isnan(stn_da_tmax.stns[BAD])
        ss_tmin = StationSelect(stn_da_tmin, mask_tmin)
        ss_tmax = StationSelect(stn_da_tmax, mask_tmax)
        self.rgn_tmin = _rgn_nnghs_keys(stn_da_tmin.stns[mask_tmin & np.isfinite(stn_da_tmin.stns[MASK])])   # :487-490
        self.rgn_tmax = _rgn_nnghs_keys(stn_da_tmax.stns[mask_tmax & np.isfinite(stn_da_tmax.stns[MASK])])
        self.interp_tmin = InterpTair(KrigTair(ss_tmin), GwrTairAnom(ss_tmin))
        self.interp_tmax = InterpTair(KrigTair(ss_tmax), GwrTairAnom(ss_tmax))
        self.a_pt = build_empty_pt()

    def interp_pt(self, fix_invalid=True, stns_rm=None):           # :526-592
        a_pt = self.a_pt
        if a_pt[CLIMDIV] not in self.rgn_tmin:                     # KeyError at :563
            raise OracleError(ST_CLIMDIV, "KeyError: %r" % a_pt[CLIMDIV])
        for m in range(1, 13):
            a_pt[lst_name(m)] = a_pt["tmin%02d" % m]               # :562
        tmin_dly, tmin_norms, tmin_se = self.interp_tmin.interp(a_pt, stns_rm=stns_rm)
        if a_pt[CLIMDIV] not in self.rgn_tmax:                     # KeyError at :572
            raise OracleError(ST_CLIMDIV, "KeyError: %r" % a_pt[CLIMDIV])
        for m in range(1, 13):
            a_pt[lst_name(m)] = a_pt["tmax%02d" % m]               # :571
        tmax_dly, tmax_norms, tmax_se = self.interp_tmax.interp(a_pt, stns_rm=stns_rm)
        ninvalid = 0
        if fix_invalid:
            tmin_dly, tmax_dly, ninvalid = tmin_tmax_fixer(tmin_dly, tmax_dly)       # :581
            if ninvalid > 0:                                       # :583-590
                tmin_n = np.take(tmin_dly, self.daysNormMask)
                tmax_n = np.take(tmax_dly, self.daysNormMask)
                with np.errstate(all="ignore"):
                    tmin_mthly = np.array([np.mean(np.take(tmin_n, a)) for a in self.yrMthsMasks])
                    tmax_mthly = np.array([np.mean(np.take(tmax_n, a)) for a in self.yrMthsMasks])
                    tmin_norms = np.array([np.mean(np.take(tmin_mthly, a)) for a in self.mth_masks])
                    tmax_norms = np.array([np.mean(np.take(tmax_mthly, a)) for a in self.mth_masks])
        return tmin_dly, tmax_dly, tmin_norms, tmax_norms, tmin_se, tmax_se, ninvalid


def quantize_daily(x):
    """step25:163-164: ``rslt[:, r, c] = np.round(dly, 2) / SCALE_FACTOR`` stored into int16
    (C truncation toward zero of a float64)."""
    return (np.round(x, 2) / np.float64(SCALE_FACTOR)).astype(np.int64).astype(np.int16)


def interp_chunk(pt_interp, wrk_chk, cells=None):
    """The per-cell loop of step25:126-175 over one work chunk ``wrk_chk`` f8[32,Y,X]
    (plane layout tiling.py:205-213 / step25:136-144).  ``cells`` optionally restricts the loop to a
    list of (r, c) so that tests can sample.  Returns the step25:71-88 result buffers + status."""
    _, Y, X = wrk_chk.shape
    ndays = pt_interp.days.size
    out = dict(tmin=np.full((ndays, Y, X), FILL_I2, dtype=np.int16), tmax=np.full((ndays, Y, X), FILL_I2, dtype=np.int16),
               tmin_norm=np.full((12, Y, X), FILL_F4, dtype=np.float32), tmax_norm=np.full((12, Y, X), FILL_F4, dtype=np.float32),
               tmin_se=np.full((12, Y, X), FILL_F4, dtype=np.float32), tmax_se=np.full((12, Y, X), FILL_F4, dtype=np.float32),
               ninvalid=np.full((Y, X), FILL_I4, dtype=np.int32), status=np.zeros((Y, X), dtype=np.uint8),
               tmin_f8={}, tmax_f8={})
    rc = cells if cells is not None else [(r, c) for r in range(Y) for c in range(X)]
    a_pt = pt_interp.a_pt
    for r, c in rc:
        if not wrk_chk[2, r, c]:                                   # step25:132
            continue
        a_pt[LAT], a_pt[LON] = wrk_chk[3, r, c], wrk_chk[4, r, c]  # step25:136-140
        a_pt[ELEV], a_pt[TDI], a_pt[CLIMDIV] = wrk_chk[5, r, c], wrk_chk[6, r, c], wrk_chk[7, r, c]
        for m in range(1, 13):                                     # step25:142-144
            a_pt["tmin%02d" % m] = wrk_chk[8 + (m - 1), r, c]
            a_pt["tmax%02d" % m] = wrk_chk[20 + (m - 1), r, c]
        try:
            tmin_dly, tmax_dly, tmin_norms, tmax_norms, tmin_se, tmax_se, ninvalid = pt_interp.interp_pt()
        except OracleError as e:                                   # step25:154-160: leave fill values
            out["status"][r, c] = e.status
            continue
        out["tmin"][:, r, c] = quantize_daily(tmin_dly)            # step25:163-172
        out["tmax"][:, r, c] = quantize_daily(tmax_dly)
        out["tmin_norm"][:, r, c] = tmin_norms
        out["tmax_norm"][:, r, c] = tmax_norms
        out["tmin_se"][:, r, c] = tmin_se
        out["tmax_se"][:, r, c] = tmax_se
        out["ninvalid"][r, c] = ninvalid
        out["tmin_f8"][(r, c)] = tmin_dly
        out["tmax_f8"][(r, c)] = tmax_dly
    return out


class XvalTairOverall(object):
    """optimize.py:547-604 leave-one-out driver for one variable."""

    def __init__(self, stn_da):
        mask_stns = np.isnan(stn_da.stns[BAD])                     # :567
        ss = StationSelect(stn_da, stn_mask=mask_stns, rm_zero_dist_stns=True)     # :569
        self.stn_da = stn_da
        self.interp_tair = InterpTair(KrigTair(ss), GwrTairAnom(ss))

    def run_interp(self, stn_id, norms_only=False):                # :579-604
        xval_stn = self.stn_da.stns[self.stn_da.stn_idxs[stn_id]].copy()
        return self.interp_tair.interp(xval_stn, stn_id, norms_only=norms_only)


class XvalTairAnom(object):
    """optimize.py:477-545: cross validation of the GWR neighbour count at one station."""

    def __init__(self, stn_da):
        mask_stns = np.isnan(stn_da.stns[BAD])                     # :497
        ss = StationSelect(stn_da, stn_mask=mask_stns, rm_zero_dist_stns=True)     # :499
        self.stn_da = stn_da
        self.gwr = GwrTairAnom(ss)

    def run_xval(self, stn_id, a_nnghs):                           # :505-545
        xval_stn = self.stn_da.stns[self.stn_da.stn_idxs[stn_id]]
        xval_obs = self.stn_da.load_obs(np.array([stn_id]))[:, 0].astype(np.float64)
        a_nnghs = np.asarray(a_nnghs)
        bias = np.zeros((a_nnghs.size, 12))
        mae, r2 = bias.copy(), bias.copy()
        for x, nnghs in enumerate(a_nnghs):
            for mth in range(1, 13):
                xval_anom = xval_obs[self.stn_da.mth_idx[mth]] - xval_stn[norm_name(mth)]
                interp_tair = self.gwr.gwr_mth(xval_stn, mth, int(nnghs), stns_rm=stn_id)
                interp_anom = interp_tair - xval_stn[norm_name(mth)]
                difs = interp_anom - xval_anom
                bias[x, mth - 1] = np.mean(difs)
                mae[x, mth - 1] = np.mean(np.abs(difs))
                r_value = np.corrcoef(interp_anom, xval_anom)[0, 1]      # = stats.linregress(...)[2] (:530)
                r2[x, mth - 1] = r_value ** 2
        return bias, mae, r2


# ------------------------------------------------------------------------------------------------
# f3  variogram fitting: R get_vario_params / krig_all (twx/interp/rpy/interp.R:54-113, 147-159, 290-428)
#     [EXT: gstat variogram(), fit.variogram(fit.method=7), predict(BLUE=TRUE)]  PARITY UNPINNED against real gstat.
VARIO_WIDTH_KM = 5.0                                   # interp.R:64 width=5
FIT_LIMIT, FIT_MAXIT = 1e-6, 200                       # gstat defaults: set(fit_limit=1e-6), set(iter=200)


def sample_variogram(H, z, cutoff, width=VARIO_WIDTH_KM):
    """gstat ``variogram(z~trend, cutoff=, width=)`` on residuals ``z`` with pair distances ``H`` (great-circle km for
    long/lat data): pairs with h <= cutoff go to lag floor(h / width); per non-empty lag: np, mean distance,
    gamma = sum (z_i - z_j)^2 / (2 np).  Returns (np, dist, gamma) for the non-empty lags in lag order."""
    n = z.size
    iu = np.triu_indices(n, 1)
    h = H[iu]
    d2 = (z[iu[0]] - z[iu[1]]) ** 2
    keep = h <= cutoff
    h, d2 = h[keep], d2[keep]
    lag = np.floor(h / width).astype(np.int64)
    nb = int(np.floor(cutoff / width)) + 1
    cnt = np.bincount(lag, minlength=nb)
    sh = np.bincount(lag, weights=h, minlength=nb)
    sg = np.bincount(lag, weights=d2, minlength=nb)
    ok = cnt > 0
    return cnt[ok].astype(np.float64), sh[ok] / cnt[ok], sg[ok] / (2.0 * cnt[ok])


def fit_exp_range(npairs, dist, gamma, nugget, sill):
    """``my.autofit.gwvario(avar, model="Exp", fix.values=c(nugget, NA, sill), fit.method=7)`` (interp.R:68,87,290-428):
    exponential model gamma(h) = nugget + psill (1 - exp(-h / range)) with nugget and psill = sill - nugget fixed, the
    range fitted by weighted least squares with weights N_j / h_j^2 (gstat fit.method 7), Gauss-Newton from
    range0 = 0.1 max(dist) (interp.R:311), steps halved while the error grows, stop when the relative change of the
    weighted SSE is below 1e-6 or after 200 iterations - continued here until the step is below 1e-10 range or no step
    lowers the SSE, then polished by up to 4 Newton steps on the gradient to the root of dS/dr (vario.cu does the same).
    Returns (nugget, psill, range) or None where the R code falls
    back to a pure nugget (fit error, negative psill or range: interp.R:69-77, 391-401)."""
    psill = sill - nugget
    if not (np.isfinite(psill) and np.isfinite(nugget)) or psill < 0 or nugget < 0:
        return None
    w = npairs / (dist * dist)

    def sse(r):
        e = gamma - (nugget + psill * (1.0 - np.exp(-dist / r)))
        return float(np.sum(w * e * e))
    r = 0.1 * float(np.max(dist))
    if not (r > 0):
        return None
    s_old = sse(r)
    gstat_done = False
    for it in range(FIT_MAXIT + 60):
        ex = np.exp(-dist / r)
        e = gamma - (nugget + psill * (1.0 - ex))
        J = -psill * ex * dist / (r * r)                    # d gamma_model / d range
        den = float(np.sum(w * J * J))
        if not (den > 0):
            return None                                    # singular fit: gstat stops with an error
        step = float(np.sum(w * J * e)) / den
        s_new = None
        for _h in range(12):
            rn = r + step
            if rn > 0:
                s_new = sse(rn)
                if s_new <= s_old:
                    break
            step *= 0.5
            s_new = None
        if s_new is None:
            break                                          # no improving step: converged at r
        small_step = abs(rn - r) <= 1e-10 * rn
        r = rn
        # gstat stops at a relative SSE change below fit_limit (or after 200 iterations); the iteration is continued to
        # the minimiser itself so that the result does not depend on where inside that tolerance band one stops
        if abs(s_old - s_new) <= FIT_LIMIT * max(s_new, 1e-300):
            gstat_done = True
        s_old = s_new
        if small_step or (it >= FIT_MAXIT and gstat_done):
            break
    # near the minimum the SSE differences are rounding noise: Newton on g(r) = sum w J e (dS/dr = -2 g), each step taken
    # only while S'' > 0 (g' < 0) and |step| <= 1e-3 r
    for _it in range(4):
        if not (np.isfinite(r) and r > 0):
            break
        ex = np.exp(-dist / r)
        e = gamma - (nugget + psill * (1.0 - ex))
        J = -psill * ex * dist / (r * r)
        dJ = psill * ex * dist * (2.0 * r - dist) / (r * r * r * r)
        g = float(np.sum(w * J * e))
        gp = float(np.sum(w * (dJ * e - J * J)))
        if not gp < 0:
            break
        step = -g / gp
        if not abs(step) <= 1e-3 * r:
            break
        r = r + step
    if not (np.isfinite(r) and r > 0):
        return None
    if nugget == 0 and psill == 0:                         # interp.R:74-77
        return None
    return nugget, psill, r


def _ols_resid(X, y):
    beta = np.linalg.solve(X.T @ X, X.T @ y)
    return y - X @ beta


def get_vario_params(ngh_lon, ngh_lat, ngh_X, ngh_y, ngh_dist):
    """R ``get_vario_params`` (interp.R:54-113): exponential variogram (nugget, psill, range) of the regression-kriging
    residuals of one neighbourhood.  ``ngh_X`` n x 4 (lon, lat, elev, lst), ``ngh_dist`` the haversine distances of the
    neighbours from the point (StationSelect.ngh_dists).  Pure nugget -> (sill, 0, 0).
    Raises OracleError(ST_SINGULAR) for fewer than 7 neighbours (at n <= 5 the five-coefficient OLS fits exactly, at
    n = 6 one degree of freedom is left) and for two neighbours at the same location (gstat puts nugget + psill at h = 0,
    so V has two equal rows), as vario.cu decides them."""
    n = ngh_lon.size
    if n < 7:
        raise OracleError(ST_SINGULAR, "fewer than 7 neighbours for the variogram")
    H = gcdist_sp(ngh_lon[:, None], ngh_lat[:, None], ngh_lon[None, :], ngh_lat[None, :])
    if np.any(H[np.triu_indices(n, 1)] == 0.0):
        raise OracleError(ST_SINGULAR, "co-located neighbours: singular covariance matrix")
    cutoff = float(np.max(ngh_dist)) * 1.4                                    # :63
    k0 = int(np.argmin(ngh_dist))                                             # centre on the nearest neighbour (exact)
    Xc = np.asarray(ngh_X, dtype=np.float64) - np.asarray(ngh_X, dtype=np.float64)[k0][None, :]
    X = np.column_stack((np.ones(n), Xc[:, 0], Xc[:, 1], Xc[:, 2] * 1e-3, Xc[:, 3] * 0.1))
    r = _ols_resid(X, ngh_y)                                                  # variogram(FORMULA, ...) works on OLS residuals
    npairs, dist, gamma = sample_variogram(H, r, cutoff)                      # :64
    sill = float(np.var(r, ddof=1))                                           # :66
    model = fit_exp_range(npairs, dist, gamma, float(np.min(gamma)), sill) if gamma.size else None      # :68
    # GLS trend with the fitted model, residuals at the stations (:79-81): predict(g, stns_ngh, BLUE=TRUE)
    if model is None:
        resid = r                                                             # V = sill I: GLS = OLS
    else:
        nug, psill, rng = model
        V = np.where(H == 0, nug + psill, psill * np.exp(-H / rng))
        V[np.diag_indices(n)] = nug + psill
        Lc = np.linalg.cholesky(V)
        Z = np.linalg.solve(Lc, np.column_stack((X, ngh_y)))
        A, b = Z[:, :-1], Z[:, -1]
        beta = np.linalg.solve(A.T @ A, A.T @ b)
        resid = ngh_y - X @ beta
    sill2 = float(np.var(resid, ddof=1))                                      # :82
    npairs, dist, gamma = sample_variogram(H, resid, cutoff)                  # :83  variogram(resid~1)
    model2 = fit_exp_range(npairs, dist, gamma, float(np.min(gamma)), sill2) if gamma.size else None    # :84
    if model2 is None:
        return sill2, 0.0, 0.0                                                # :86-93,103-107
    return model2


class BuildKrigParams(object):
    """interp_tair.py:612-698: variogram parameters of a point and month with the smoothed optimal neighbour count."""

    def __init__(self, stn_slct):
        self.stn_slct = stn_slct

    def get_krig_params(self, pt, mth, rm_stnid=None, nnghs=None):
        ss = self.stn_slct
        if nnghs is None:                                                      # :666-678
            ss.set_ngh_stns(pt[LAT], pt[LON], DFLT_INIT_NNGHS, load_obs=False)
            fin = np.isfinite(ss.ngh_stns[optim_name(mth)])
            if fin.sum() == 0:
                raise OracleError(ST_NO_NNGHS, "Cannot determine the optimal # of neighbors to use!")
            nnghs = int(np.round(np.average(ss.ngh_stns[optim_name(mth)][fin], weights=ss.ngh_wgt[fin])))
        ss.set_ngh_stns(pt[LAT], pt[LON], nnghs, load_obs=False, stns_rm=rm_stnid)    # :681 (rm_stnid unused there)
        nghs = ss.ngh_stns
        X = np.column_stack([nghs[LON], nghs[LAT], nghs[ELEV], nghs[lst_name(mth)]])
        return get_vario_params(nghs[LON], nghs[LAT], X, nghs[norm_name(mth)], ss.ngh_dists)


class KrigTairAll(object):
    """interp_tair.py:700-768 + R krig_all (interp.R:147-159): variogram fit and regression kriging in one step."""

    def __init__(self, stn_slct):
        self.stn_slct = stn_slct

    def krigall(self, pt, nnghs, stns_rm=None):
        ss = self.stn_slct
        ss.set_ngh_stns(pt[LAT], pt[LON], nnghs, load_obs=False, stns_rm=stns_rm)
        nghs = ss.ngh_stns
        interp_norms = np.zeros(12)
        self.last_vario = np.zeros((12, 3))
        for mth in range(1, 13):
            X = np.column_stack([nghs[LON], nghs[LAT], nghs[ELEV], nghs[lst_name(mth)]])
            y = nghs[norm_name(mth)]
            nug, psill, rng = get_vario_params(nghs[LON], nghs[LAT], X, y, ss.ngh_dists)
            x = np.array([pt[LON], pt[LAT], pt[ELEV], pt[lst_name(mth)]], dtype=np.float64)
            mean, var = ked_gstat(nghs[LON], nghs[LAT], X, y, pt[LON], pt[LAT], x, nug, psill, rng)
            interp_norms[mth - 1] = mean
            self.last_vario[mth - 1] = (nug, psill, rng)
        return interp_norms


class XvalTairNorm(object):
    """optimize.py:210-266: leave-one-out error of the kriged normals for a set of neighbour counts."""

    def __init__(self, stn_da):
        mask_stns = np.isnan(stn_da.stns[BAD])
        ss = StationSelect(stn_da, stn_mask=mask_stns, rm_zero_dist_stns=True)
        self.krig = KrigTairAll(ss)
        self.stn_da = stn_da

    def run_xval(self, stn_id, abw_nngh):
        xval_stn = self.stn_da.stns[self.stn_da.stn_idxs[stn_id]]
        err = np.zeros((12, len(abw_nngh)))
        xval_norms = np.array([xval_stn[norm_name(m)] for m in range(1, 13)])
        for x, bw in enumerate(abw_nngh):
            err[:, x] = self.krig.krigall(xval_stn, int(bw), stns_rm=stn_id) - xval_norms
        return err

'''
Classes and functions for performing Tair interpolation: the `twx.interp.interp_tair` interface
(twx/interp/interp_tair.py) with every numerical stage running on the GPU through libtwxi.

Kept, with the reference's signatures: KrigTair, GwrTairAnom, InterpTair, PtInterpTair, StationDataWrkChk,
build_empty_pt (tmin_tmax_fixer runs inside the CUDA library: twxi_interp_cells / twxi_interp_chunk).  New batch entry points (no reference equivalent): InterpTair.interp_batch,
PtInterpTair.interp_chunk.  KrigTairAll / BuildKrigParams run the variogram fitting of R get_vario_params as a CUDA
kernel; PredictorGrids / interp_to_lonlat read the rasters of a PredictorStore.  Not rebuilt: GwrTairAnomR, GwrTairNorm
(dead code in the reference).
'''

__all__ = ["GwrTairAnom", 'KrigTair', 'KrigTairAll', 'BuildKrigParams', 'InterpTair', 'StationDataWrkChk', 'PtInterpTair',
           'RecordStream', 'PredictorGrids']

import numpy as np

from .station_select import StationSelect
from ..db import LON, LAT, ELEV, TDI, LST, BAD, MASK, CLIMDIV, YEAR, MONTH, STN_ID, \
    StationSerialDataDb, get_norm_varname, get_optim_varname, get_lst_varname, get_optim_anom_varname
from .. import _lib
from .. import context as _context

KRIG_TREND_VARS = (LON, LAT, ELEV, LST)
GWR_TREND_VARS = (LON, LAT, ELEV, TDI, LST)
LST_TMAX = 'lst_tmax'
LST_TMIN = 'lst_tmin'
DFLT_INIT_NNGHS = 100
_CI_CRITVAL = -1.959963984540054        # scipy.stats.norm.ppf(0.025) (interp_tair.py:792)


def _raise_status(st):
    st = int(st)
    if st == _lib.ST_OK:
        return
    if st == _lib.ST_TOO_FEW_STNS:
        raise IndexError(_lib.STATUS_MESSAGES[st])
    if st == _lib.ST_CLIMDIV:
        raise KeyError(_lib.STATUS_MESSAGES[st])
    if st == _lib.ST_SINGULAR:
        raise FloatingPointError(_lib.STATUS_MESSAGES[st])
    raise Exception(_lib.STATUS_MESSAGES.get(st, "interpolation failed (status %d)" % st))


def _pt_lst(pt):
    return np.array([pt[get_lst_varname(m)] for m in range(1, 13)], dtype=np.float64)


def build_empty_pt():
    ptDtype = [(LON, np.float64), (LAT, np.float64), (ELEV, np.float64),
               (TDI, np.float64), (CLIMDIV, np.float64), (MASK, np.float64)]
    ptDtype.extend([("tmin%02d" % mth, np.float64) for mth in np.arange(1, 13)])
    ptDtype.extend([("tmax%02d" % mth, np.float64) for mth in np.arange(1, 13)])
    ptDtype.extend([(get_norm_varname(mth), np.float64) for mth in np.arange(1, 13)])
    ptDtype.extend([(get_optim_varname(mth), np.float64) for mth in np.arange(1, 13)])
    ptDtype.extend([(get_lst_varname(mth), np.float64) for mth in np.arange(1, 13)])
    ptDtype.extend([(get_optim_anom_varname(mth), np.float64) for mth in np.arange(1, 13)])
    a_pt = np.empty(1, dtype=ptDtype)
    return a_pt[0]


class PredictorGrids(object):
    '''
    Auxiliary predictor values of a point from the predictor rasters (interp_tair.py:87-141).  The reference opens one
    netCDF file per predictor; here the rasters are a `PredictorStore` (topowx_b200/interp/feed.py: .npy rasters, or the
    path of such a directory).  Order 0 (default) takes the value of the grid cell that contains the point and, with
    chgLatLon, moves the point to the cell centre; order 1 interpolates bilinearly and falls back to the nearest cell where
    a corner is missing (the bm.interp(order=1) -> order=0 fallback of :131-139).
    '''
    PT_FIELD = {'elev': ELEV, 'tdi': TDI, 'climdiv': CLIMDIV, 'mask': MASK}

    def __init__(self, store, interpOrders=None):
        from .feed import PredictorStore, PLANE_NAMES
        self.store = store if isinstance(store, PredictorStore) else PredictorStore(store)
        self.names = ['mask'] + list(PLANE_NAMES)
        self.rasters = dict(zip(PLANE_NAMES, self.store.rasters))
        self.rasters['mask'] = self.store.variables['mask']
        orders = {} if interpOrders is None else dict(interpOrders)
        self.orders = {n: int(orders.get(n, 0)) for n in self.names}
        self.lons = np.asarray(self.store.variables['lon'], dtype=np.float64)
        self.lats = np.asarray(self.store.variables['lat'], dtype=np.float64)          # descending
        self.dx = float(self.lons[1] - self.lons[0])
        self.dy = float(self.lats[0] - self.lats[1])

    def get_row_col(self, lon, lat):
        col = int(np.floor((lon - (self.lons[0] - 0.5 * self.dx)) / self.dx))
        row = int(np.floor(((self.lats[0] + 0.5 * self.dy) - lat) / self.dy))
        if not (0 <= row < self.lats.size and 0 <= col < self.lons.size):
            raise Exception("Lon/Lat outside the bounds of the predictor grids")      # GeoNc.get_row_col
        return row, col, float(self.lons[col]), float(self.lats[row])

    def _bilinear(self, a, lon, lat):
        fx = (lon - self.lons[0]) / self.dx
        fy = (self.lats[0] - lat) / self.dy
        c0, r0 = int(np.floor(fx)), int(np.floor(fy))
        if not (0 <= r0 < self.lats.size - 1 and 0 <= c0 < self.lons.size - 1):
            return np.nan
        tx, ty = fx - c0, fy - r0
        v = np.asarray(a[r0:r0 + 2, c0:c0 + 2], dtype=np.float64)
        return float((1 - ty) * ((1 - tx) * v[0, 0] + tx * v[0, 1]) + ty * ((1 - tx) * v[1, 0] + tx * v[1, 1]))

    def setPtValues(self, aPt, chgLatLon=True):
        row, col, gridlon, gridlat = self.get_row_col(float(aPt[LON]), float(aPt[LAT]))
        for n in self.names:
            field = self.PT_FIELD.get(n, n)
            if self.orders[n] == 1 and not chgLatLon:
                v = self._bilinear(self.rasters[n], float(aPt[LON]), float(aPt[LAT]))
                if not np.isfinite(v):
                    v = float(self.rasters[n][row, col])
            else:
                v = float(self.rasters[n][row, col])
            aPt[field] = v
        if chgLatLon:
            aPt[LON], aPt[LAT] = gridlon, gridlat


class GwrTairAnom(object):
    '''
    Geographically weighted regression interpolation of daily temperature anomalies for a month
    (interp_tair.py:215-314).
    '''

    def __init__(self, stn_slct):
        self.stn_slct = stn_slct

    def gwr_mth(self, pt, mth, nnghs=None, stns_rm=None):
        '''
        Interpolates the daily anomalies of month `mth` with GWR, adds them to pt's monthly normal
        (pt[normMM]) and returns the daily values of that month (interp_tair.py:261-314).
        '''
        ss = self.stn_slct
        ctx = ss.ctx
        vals, st = ctx.gwr_mth(pt[LAT], pt[LON], pt[ELEV], pt[TDI], _pt_lst(pt), int(mth),
                               pt[get_norm_varname(mth)], nnghs=nnghs, rm_idx=ctx.rm_indices(stns_rm),
                               rm_zero=ss.rm_zero_dist_stns)
        _raise_status(st[0])
        return vals[0]


class KrigTair(object):
    '''
    Moving window regression kriging of monthly normals with variogram parameters passed in or smoothed
    from the neighboring stations (interp_tair.py:770-926).  The R/gstat call is replaced by the CUDA
    kriging-with-external-drift kernel.
    '''

    def __init__(self, stn_slct):
        self.stn_slct = stn_slct
        self.ci_critval = _CI_CRITVAL

    def std_err_ci(self, tair_mean, tair_var):
        std_err = np.sqrt(tair_var) if tair_var >= 0 else 0
        ci_r = np.abs(std_err * self.ci_critval)
        return std_err, (tair_mean - ci_r, tair_mean + ci_r)

    def krig(self, pt, mth, nnghs=None, vario_params=None, stns_rm=None):
        '''
        Returns (tair_mean, tair_var) for month `mth` at `pt` (interp_tair.py:853-926).
        '''
        ss = self.stn_slct
        ctx = ss.ctx
        mean, var, st = ctx.krig(pt[LAT], pt[LON], pt[ELEV], _pt_lst(pt), mth=int(mth), nnghs=nnghs,
                                 vario=vario_params, rm_idx=ctx.rm_indices(stns_rm), rm_zero=ss.rm_zero_dist_stns)
        _raise_status(st[0])
        return float(mean[0, 0]), float(var[0, 0])


class BuildKrigParams(object):
    '''
    Moving window regression kriging variogram parameters for a specific point (interp_tair.py:612-698): the R
    function get_vario_params (gstat variogram + fit.variogram, interp.R:54-113) runs as a CUDA kernel (twxi_fit_vario).
    '''

    def __init__(self, stn_slct):
        self.stn_slct = stn_slct

    def get_krig_params(self, pt, mth, rm_stnid=None):
        '''
        Returns (nug, psill, rng) of the exponential variogram for month `mth` at `pt`, with the smoothed optimal
        number of neighbours.  Like the reference (:681), `rm_stnid` is accepted but not applied to the neighbour search.
        '''
        ss = self.stn_slct
        vario, st = ss.ctx.fit_vario(pt[LAT], pt[LON], mth=int(mth), rm_zero=ss.rm_zero_dist_stns)
        _raise_status(st[0])
        return float(vario[0, 0, 0]), float(vario[0, 0, 1]), float(vario[0, 0, 2])

    def get_krig_params_batch(self, lat, lon, nnghs=None, rm_idx=None):
        '''Batch form (new): all 12 months for arrays of points -> vario [n, 12, 3], status [n].'''
        ss = self.stn_slct
        return ss.ctx.fit_vario(lat, lon, mth=0, nnghs=nnghs, rm_idx=rm_idx, rm_zero=ss.rm_zero_dist_stns)


class KrigTairAll(object):
    '''
    Moving window variogram fitting and regression kriging of monthly normals all in one step (interp_tair.py:700-768,
    R krig_all interp.R:147-159); used to optimise the local number of neighbouring stations (step 21).
    '''

    def __init__(self, stn_slct):
        self.stn_slct = stn_slct

    def krigall(self, pt, nnghs, stns_rm=None):
        '''Returns the 12 interpolated monthly normals at `pt` using `nnghs` neighbours.'''
        ss = self.stn_slct
        ctx = ss.ctx
        mean, var, vario, st = ctx.krig_all(pt[LAT], pt[LON], pt[ELEV], _pt_lst(pt), int(nnghs),
                                            rm_idx=ctx.rm_indices(stns_rm), rm_zero=ss.rm_zero_dist_stns)
        _raise_status(st[0])
        return mean[0]


class InterpTair(object):
    '''
    Monthly normals (moving window regression kriging) and daily temperatures (GWR) for a single
    temperature variable (interp_tair.py:371-439).
    '''

    def __init__(self, krig_tair, gwr_tair):
        self.krig_tair = krig_tair
        self.gwr_tair = gwr_tair
        self.mth_masks = self.gwr_tair.stn_slct.stn_da.mth_idx
        self.ndays = self.gwr_tair.stn_slct.stn_da.days.size

    def interp(self, pt, stns_rm=None):
        '''
        Returns (tair_daily[ndays], tair_norms[12], tair_se[12]); like the reference it also stores the
        kriged normals in pt[normMM] (interp_tair.py:433).
        '''
        ss = self.gwr_tair.stn_slct
        ctx = ss.ctx
        dly, norms, se, var, st = ctx.interp_points(pt[LAT], pt[LON], pt[ELEV], pt[TDI], _pt_lst(pt),
                                                    rm_idx=ctx.rm_indices(stns_rm), rm_zero=ss.rm_zero_dist_stns)
        _raise_status(st[0])
        for mth in range(1, 13):
            pt[get_norm_varname(mth)] = norms[0, mth - 1]
        return dly[0], norms[0], se[0]

    def interp_batch(self, lat, lon, elev, tdi, lst, rm_idx=None, daily=True):
        '''
        Batch form (new): arrays of points, lst [npts, 12]; rm_idx [npts, n_rm] indices into the selected
        stations (-1 = none).  Returns (daily [npts, ndays] or None, norms, se, var [npts, 12], status [npts]).
        '''
        ss = self.gwr_tair.stn_slct
        return ss.ctx.interp_points(lat, lon, elev, tdi, lst, rm_idx=rm_idx, rm_zero=ss.rm_zero_dist_stns,
                                    daily=daily)


class PtInterpTair(object):
    '''
    Monthly normals and daily temperatures for both Tmin and Tmax (interp_tair.py:441-592).
    '''

    def __init__(self, stn_da_tmin, stn_da_tmax, aux_fpaths=None, interp_orders=None, norms_only=False, device=0):
        self.days = stn_da_tmin.days
        self.stn_da_tmin = stn_da_tmin
        self.stn_da_tmax = stn_da_tmax
        daysNormMask = np.nonzero(np.logical_and(self.days[YEAR] >= 1981, self.days[YEAR] <= 2010))[0]
        if daysNormMask.size == 0:
            raise IndexError("the observation record has no day within 1981-2010")   # uYrs[0], interp_tair.py:470
        self.daysNormMask = daysNormMask
        mask_stns_tmin = np.isnan(stn_da_tmin.stns[BAD])
        mask_stns_tmax = np.isnan(stn_da_tmax.stns[BAD])
        stn_slct_tmin = StationSelect(stn_da_tmin, mask_stns_tmin, device=device)
        stn_slct_tmax = StationSelect(stn_da_tmax, mask_stns_tmax, device=device)
        self.interp_tmin = InterpTair(KrigTair(stn_slct_tmin), GwrTairAnom(stn_slct_tmin))
        self.interp_tmax = InterpTair(KrigTair(stn_slct_tmax), GwrTairAnom(stn_slct_tmax))
        self.ctx_tmin = stn_slct_tmin.ctx
        self.ctx_tmax = stn_slct_tmax.ctx
        self.norms_only = norms_only
        self.pGrids = None
        if aux_fpaths is not None:                                 # a PredictorStore or the path of one (feed.py)
            self.pGrids = PredictorGrids(aux_fpaths, interp_orders)
        self.a_pt = build_empty_pt()

    def interp_to_lonlat(self, lon, lat, fixInvalid=True, chgLatLon=True, stns_rm=None, elev=None):
        '''
        Interpolate Tmin and Tmax to a lon/lat; the auxiliary predictors come from the predictor rasters
        (interp_tair.py:513-524).  Returns the 7-tuple of interp_pt.
        '''
        if self.pGrids is None:
            raise Exception("PtInterpTair was built without predictor rasters (aux_fpaths)")
        self.a_pt[LON] = lon
        self.a_pt[LAT] = lat
        self.pGrids.setPtValues(self.a_pt, chgLatLon)
        if elev is not None:
            self.a_pt[ELEV] = elev
        if self.a_pt[MASK] == 0:
            raise Exception('Point is outside interpolation region')
        return self.interp_pt(fixInvalid, stns_rm)

    def interp_pt(self, fix_invalid=True, stns_rm=None):
        '''
        Interpolate daily and monthly normal Tmin and Tmax for the current PtInterpTair.a_pt
        (interp_tair.py:526-592).  Returns (tmin_dly, tmax_dly, tmin_norms, tmax_norms, tmin_se, tmax_se,
        ninvalid).
        '''
        a_pt = self.a_pt
        lst_tmin = np.array([a_pt["tmin%02d" % m] for m in range(1, 13)], dtype=np.float64)
        lst_tmax = np.array([a_pt["tmax%02d" % m] for m in range(1, 13)], dtype=np.float64)
        # stns_rm names stations by id; each variable's context has its own index for them (interp_tair.py:565,574)
        rm_a = self.ctx_tmin.rm_indices(stns_rm)
        rm_b = self.ctx_tmax.rm_indices(stns_rm)
        r = _context.interp_cells(self.ctx_tmin, self.ctx_tmax, a_pt[LAT], a_pt[LON], a_pt[ELEV], a_pt[TDI],
                                  a_pt[CLIMDIV], lst_tmin, lst_tmax, rm_idx_tmin=rm_a, rm_idx_tmax=rm_b,
                                  fix_invalid=fix_invalid)
        tmin, tmax, nmin, nmax, semin, semax, ninv, st = r
        _raise_status(st[0])
        for m in range(1, 13):                                    # side effects of the reference (:562-575, :433)
            a_pt[get_lst_varname(m)] = a_pt["tmax%02d" % m]
            a_pt[get_norm_varname(m)] = nmax[0, m - 1]
        return tmin[0], tmax[0], nmin[0], nmax[0], semin[0], semax[0], int(ninv[0]) if fix_invalid else 0

    def interp_chunk(self, wrk_chk, out=None, wait=True):
        '''
        Batch form (new): one work chunk f8[32, ny, nx] exactly as Tiler.next() builds it (tiling.py:205-213);
        replaces the per-cell loop of step25_mpi_interp_tair.py:126-175.  Returns the step25 result buffers
        (tmin/tmax int16 [ndays, ny, nx], *_norm/*_se float32 [12, ny, nx], ninvalid int32, status uint8).
        wait=False submits the chunk and returns at once (pinned wrk_chk / out buffers; the results are valid after
        interp_chunk_wait), the way the worker loop hands a chunk to the writer while it computes the next
        (step25:176-196).
        '''
        return _context.interp_chunk(self.ctx_tmin, self.ctx_tmax, wrk_chk, out=out, daily=not self.norms_only, wait=wait)

    def interp_chunk_wait(self):
        '''Completion of the chunks submitted with interp_chunk(..., wait=False).'''
        _context.interp_chunk_wait(self.ctx_tmin)

    def interp_chunk_stream(self, wrk_chk, months=False):
        '''
        New: interp_chunk over a long record in day windows (twxi_tile_begin / _days / _end).  The kriging and the GWR hat
        rows run once here; the returned RecordStream emits the record window by window, so the device holds one window of
        dailies instead of the whole record.  The windows concatenate to exactly the bytes interp_chunk returns.  One
        stream per context pair at a time: a new stream discards an open one.  months=True: every window also returns the
        monthly means of the months it completes (twxi_tile_days_mth), so one pass emits dailies, normals and monthly grids.
        '''
        return RecordStream(self, wrk_chk, months)


class RecordStream(object):
    '''
    The daily record of one work chunk in consecutive windows (PtInterpTair.interp_chunk_stream).  `day0` is the first day
    the next window starts at; `days(n)` returns {tmin, tmax} int16 [n, ny, nx]; `years()` yields (day0, out) per calendar
    year of the remaining days; `finish()` returns the normals, se, ninvalid and status of interp_chunk and closes the
    stream.  Buffers live where wrk_chk lives (numpy on the host, torch tensors on its CUDA device).  With months=True
    each window's dict also holds tmin_mth, tmax_mth float32 [nmth, ny, nx] and mth_groups [(year, month, ndays)] of the
    months that end in it (context.tile_days_mth).
    '''

    def __init__(self, pt_interp, wrk_chk, months=False):
        self.ctx_tmin, self.ctx_tmax = pt_interp.ctx_tmin, pt_interp.ctx_tmax
        self.days_meta = pt_interp.days
        self.device = wrk_chk.device if _lib.is_device(wrk_chk) else None
        self.shape = _context.tile_begin(self.ctx_tmin, self.ctx_tmax, wrk_chk)
        self.groups = _context.MonthGroups(self.days_meta) if months else None
        self.day0 = 0

    def days(self, n, out=None):
        if self.groups is None:
            o = _context.tile_days(self.ctx_tmin, self.ctx_tmax, n, self.shape, out=out, device=self.device)
        else:
            o = _context.tile_days_mth(self.ctx_tmin, self.ctx_tmax, n, self.shape, self.groups, out=out,
                                       device=self.device)
        self.day0 += int(n)
        return o

    def years(self):
        yrs = np.asarray(self.days_meta[YEAR])
        while self.day0 < yrs.size:
            d0 = self.day0
            n = int(np.searchsorted(yrs, yrs[d0], side="right")) - d0
            yield d0, self.days(n)

    def finish(self, out=None):
        return _context.tile_end(self.ctx_tmin, self.ctx_tmax, self.shape, out=out, device=self.device)


class StationDataWrkChk(StationSerialDataDb):
    '''
    StationSerialDataDb wrapper that preloads and caches all station observations within a lon/lat bounding box
    (interp_tair.py:997-1097), with the reference's contract: `set_obs` caches the columns of the stations inside the box
    +/- deg_buf split by month, `load_obs(ids, mth)` returns them in DB order and grows the buffer by one degree until
    every requested station is found.  The GPU path does not need it (the whole observation table is resident in HBM,
    twxi_ctx_set_obs); it serves host-side callers written against the reference.
    '''

    def __init__(self, nc_path, var_name, vcc_size=None, vcc_nelems=None, vcc_preemption=None):
        StationSerialDataDb.__init__(self, nc_path, var_name, vcc_size, vcc_nelems, vcc_preemption)
        self.chk_stnids = None
        self.chk_obs = None
        self.chk_deg_buf = None
        self.chk_bnds = None

    def set_obs(self, bnds, deg_buf=3):
        minLat, maxLat = bnds[0] - deg_buf, bnds[1] + deg_buf
        minLon, maxLon = bnds[2] - deg_buf, bnds[3] + deg_buf
        maskStns = np.logical_and(np.logical_and(self.stns[LAT] >= minLat, self.stns[LAT] <= maxLat),
                                  np.logical_and(self.stns[LON] >= minLon, self.stns[LON] <= maxLon))
        maskStns = np.nonzero(maskStns)[0]
        self.chk_stnids = np.take(self.stn_ids, maskStns)
        achkObs = self.var[:, maskStns]
        self.chk_obs = {mth: np.take(achkObs, self.mth_idx[mth], axis=0) for mth in range(1, 13)}
        self.chk_deg_buf = deg_buf
        self.chk_bnds = bnds

    def load_obs(self, stn_ids, mth=None):
        if mth is None:
            return StationSerialDataDb.load_obs(self, stn_ids, mth)
        if self.chk_obs is None:
            raise Exception("set_obs has not been called")
        stn_ids = np.atleast_1d(stn_ids)
        mask = np.nonzero(np.isin(self.chk_stnids, stn_ids))[0]
        while mask.size != stn_ids.size:                          # :1089-1093 "Increasing obs chunk..."
            if self.chk_stnids.size == self.stn_ids.size:
                raise KeyError("station id not in the database")
            self.set_obs(self.chk_bnds, self.chk_deg_buf + 1)
            mask = np.nonzero(np.isin(self.chk_stnids, stn_ids))[0]
        return np.take(self.chk_obs[mth], mask, axis=1)

'''
Cross validation of the full interpolation: the `XvalTairOverall` interface of twx/interp/optimize.py:547-604
(the driver class of scripts/step24_mpi_xval_interp.py) on the GPU path, and `XvalTairAnom` (optimize.py:477-545, the
driver class of scripts/step23: cross validation of the GWR neighbour count), which is the same GWR kernel with the
neighbour count overridden (SURVEY §8f rank 2); `XvalTairNorm` (optimize.py:210-266, step 21) and `StationKrigParams`
(optimize.py:408-474, step 22) run the variogram fitting of R get_vario_params as a CUDA kernel (SURVEY §8f rank 3).
'''

__all__ = ['XvalTairOverall', 'XvalTairAnom', 'XvalTairNorm', 'StationKrigParams', 'build_nstn_bandwidths']

import numpy as np

from ..db import BAD, STN_ID, LAT, LON, ELEV, TDI, StationSerialDataDb, get_lst_varname, get_norm_varname
from .station_select import StationSelect
from .interp_tair import KrigTair, GwrTairAnom, InterpTair, KrigTairAll, BuildKrigParams, _raise_status


class XvalTairOverall():
    '''
    Leave-one-out cross validation of interpolated monthly normals and daily temperatures using previously
    optimized variogram and number-of-stations parameters.
    '''

    def __init__(self, path_db, tair_var, device=0):
        '''
        path_db : str or StationSerialDataDb
            Serially complete station database (path, or an already opened database).
        tair_var : str
            'tmin' or 'tmax'
        '''
        stn_da = path_db if isinstance(path_db, StationSerialDataDb) else StationSerialDataDb(path_db, tair_var)
        mask_stns = np.isnan(stn_da.stns[BAD])
        stn_slct = StationSelect(stn_da, stn_mask=mask_stns, rm_zero_dist_stns=True, device=device)
        krig_tair = KrigTair(stn_slct)
        gwr_tair = GwrTairAnom(stn_slct)
        self.stn_da = stn_da
        self.interp_tair = InterpTair(krig_tair, gwr_tair)
        self.mth_masks = stn_da.mth_idx

    def run_interp(self, stn_id):
        '''
        Leave-one-out interpolation at one station: returns (tair_daily, tair_norms[12], tair_se[12])
        (optimize.py:579-604).
        '''
        xval_stn = self.stn_da.stns[self.stn_da.stn_idxs[stn_id]]
        return self.interp_tair.interp(xval_stn, xval_stn[STN_ID])

    def run_interp_batch(self, stn_ids, daily=True):
        '''
        Batch form (new): all stations of `stn_ids` in one GPU call.  Returns (daily [n, ndays] or None,
        norms [n, 12], se [n, 12], status [n]); stations that fail keep fill values, as the step24 worker
        does on an exception (step24_mpi_xval_interp.py:59-65).
        '''
        ctx = self.interp_tair.gwr_tair.stn_slct.ctx
        rows = np.array([self.stn_da.stn_idxs[s] for s in stn_ids])
        s = self.stn_da.stns[rows]
        lst = np.stack([s[get_lst_varname(m)] for m in range(1, 13)], axis=1)
        rm = ctx.local_of_db[rows].astype(np.int32).reshape(-1, 1)
        dly, norms, se, var, st = self.interp_tair.interp_batch(s[LAT], s[LON], s[ELEV], s[TDI], lst, rm_idx=rm,
                                                                 daily=daily)
        return dly, norms, se, st

    def run_xval(self, stn_id):
        '''
        Leave-one-out skill at one station: (bias, mae, r2), each [12], of the interpolated daily series against the
        station's own observations (the statistics of XvalTairAnom.run_xval, optimize.py:520-531, over the full series).
        '''
        bias, mae, r2, norms, se, st = self.run_xval_batch([stn_id])
        _raise_status(st[0])
        return bias[0], mae[0], r2[0]

    def run_xval_batch(self, stn_ids, daily=False):
        '''
        Batch form (new): leave-one-out interpolation and its skill at every station of `stn_ids` in one library call
        (twxi_xval_overall: the statistics are computed on the device, and the daily series leave it only with `daily`).
        Returns (bias, mae, r2, norms, se [n, 12], status [n]) and, with `daily`, the dailies [n, ndays] of
        run_interp_batch; failed stations have NaN statistics and fill values elsewhere.
        '''
        ctx = self.interp_tair.gwr_tair.stn_slct.ctx
        rows = np.array([self.stn_da.stn_idxs[s] for s in stn_ids], dtype=np.int64)
        loc = ctx.local_of_db[rows]
        if np.any(loc < 0):
            raise KeyError("station is not among the selected (good) stations")
        bias, mae, r2, norms, se, st, dly = ctx.xval_overall(loc.astype(np.int32), daily=daily)
        return (bias, mae, r2, norms, se, st, dly) if daily else (bias, mae, r2, norms, se, st)


def build_nstn_bandwidths(rng_min, rng_max, pct_step):
    '''
    Range of neighbour-count bandwidths within [rng_min, rng_max] with fractional spacing pct_step
    (optimize.py:376-405; build_nstn_bandwidths(35, 150, 0.10) is the 16-value set used by steps 21 and 23).
    '''
    min_nghs = []
    n = rng_min
    while n <= rng_max:
        min_nghs.append(n)
        n = n + np.round(pct_step * n)
    return np.array(min_nghs, dtype=int)


def _linregress_r(x, y):
    """Pearson r = scipy.stats.linregress(x, y)[2] (optimize.py:530) without importing scipy."""
    xm, ym = x - x.mean(), y - y.mean()
    den = np.sqrt((xm * xm).sum() * (ym * ym).sum())
    return (xm * ym).sum() / den if den > 0 else 0.0


class XvalTairAnom(object):
    '''
    Cross validation to optimize the local number of neighboring stations used by the geographically weighted
    regression of daily temperature anomalies (optimize.py:477-545).
    '''

    def __init__(self, path_db, tair_var, device=0):
        stn_da = path_db if isinstance(path_db, StationSerialDataDb) else StationSerialDataDb(path_db, tair_var)
        mask_stns = np.isnan(stn_da.stns[BAD])
        stn_slct = StationSelect(stn_da, stn_mask=mask_stns, rm_zero_dist_stns=True, device=device)
        self.stn_da = stn_da
        self.gwr = GwrTairAnom(stn_slct)

    def run_xval(self, stn_id, a_nnghs):
        '''
        Leave-one-out GWR at one station for every neighbour count of `a_nnghs`: returns (bias, mae, r2), each
        [len(a_nnghs), 12] (optimize.py:505-545).
        '''
        bias, mae, r2, st = self.run_xval_batch([stn_id], a_nnghs)
        _raise_status(st[0])
        return bias[0], mae[0], r2[0]

    def run_xval_batch(self, stn_ids, a_nnghs):
        '''
        Batch form (new): every station of `stn_ids` x every neighbour count x 12 months in ONE library call
        (twxi_xval_anom: the neighbour search runs once per station, the counts and months loop on the device).
        Returns bias, mae, r2 [n, len(a_nnghs), 12] and status [n] (failed stations keep NaN).
        '''
        ctx = self.gwr.stn_slct.ctx
        rows = np.array([self.stn_da.stn_idxs[s] for s in stn_ids])
        loc = ctx.local_of_db[rows]
        if np.any(loc < 0):
            raise KeyError("station is not among the selected (good) stations")
        return ctx.xval_anom(loc.astype(np.int32), np.asarray(a_nnghs, dtype=np.int32))


class XvalTairNorm(object):
    '''
    Cross validation to optimize the local number of neighboring stations used for moving window regression kriging of
    monthly temperature normals (optimize.py:210-266).
    '''

    def __init__(self, path_db, tair_var, device=0):
        stn_da = path_db if isinstance(path_db, StationSerialDataDb) else StationSerialDataDb(path_db, tair_var)
        mask_stns = np.isnan(stn_da.stns[BAD])
        stn_slct = StationSelect(stn_da, stn_mask=mask_stns, rm_zero_dist_stns=True, device=device)
        self.krig = KrigTairAll(stn_slct)
        self.stn_da = stn_da

    def run_xval(self, stn_id, abw_nngh):
        '''Leave-one-out errors (modeled - observed normal) [12, len(abw_nngh)] at one station (optimize.py:239-266).'''
        err, st = self.run_xval_batch([stn_id], abw_nngh)
        _raise_status(st[0])
        return err[0]

    def run_xval_batch(self, stn_ids, abw_nngh):
        '''
        Batch form (new): every station of `stn_ids` x every bandwidth in one library call (twxi_krig_all over
        len(stn_ids) * len(abw_nngh) points).  Returns err [n, 12, len(abw_nngh)] (NaN where a fit or a system fails)
        and status [n] (first failure per station).
        '''
        ss = self.krig.stn_slct
        ctx = ss.ctx
        abw = np.asarray(abw_nngh, dtype=np.int32)
        rows = np.array([self.stn_da.stn_idxs[s] for s in stn_ids])
        s = self.stn_da.stns[rows]
        n, nb = rows.size, abw.size
        rep = lambda a: np.repeat(np.asarray(a), nb, axis=0)
        lst = np.stack([s[get_lst_varname(m)] for m in range(1, 13)], axis=1)
        rm = ctx.local_of_db[rows].astype(np.int32).reshape(-1, 1)
        mean, var, vario, st = ctx.krig_all(rep(s[LAT]), rep(s[LON]), rep(s[ELEV]), rep(lst), np.tile(abw, n),
                                            rm_idx=rep(rm), rm_zero=ss.rm_zero_dist_stns)
        norms = np.stack([s[get_norm_varname(m)] for m in range(1, 13)], axis=1)           # [n, 12]
        mean = mean.reshape(n, nb, 12)
        st = st.reshape(n, nb)
        err = np.where((st == 0)[:, :, None], mean - norms[:, None, :], np.nan).transpose(0, 2, 1)
        first = np.array([next((int(v) for v in row if v != 0), 0) for row in st], dtype=np.uint8)
        return err, first


class StationKrigParams(object):
    '''
    Moving window regression kriging variogram parameters at station locations, once the optimal station bandwidths
    have been set (optimize.py:408-474, step 22).
    '''

    def __init__(self, path_db, tair_var, device=0):
        stn_da = path_db if isinstance(path_db, StationSerialDataDb) else StationSerialDataDb(path_db, tair_var)
        mask_stns = np.isnan(stn_da.stns[BAD])
        stn_slct = StationSelect(stn_da, stn_mask=mask_stns, rm_zero_dist_stns=False, device=device)
        self.stn_da = stn_da
        self.krigparams = BuildKrigParams(stn_slct)

    def get_krig_params(self, stn_id):
        '''Returns (nugs, psills, rngs), each [12], at one station (optimize.py:438-474).'''
        v, st = self.get_krig_params_batch([stn_id])
        _raise_status(st[0])
        return v[0, :, 0], v[0, :, 1], v[0, :, 2]

    def get_krig_params_batch(self, stn_ids):
        '''Batch form (new): vario [n, 12, 3] and status [n] for many stations in one library call.'''
        rows = np.array([self.stn_da.stn_idxs[s] for s in stn_ids])
        s = self.stn_da.stns[rows]
        return self.krigparams.get_krig_params_batch(s[LAT], s[LON])

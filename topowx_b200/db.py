"""Station-database containers for the interpolation hot path.

Mirrors the part of ``twx.db`` that ``twx.interp`` consumes (``twx/db/station_data.py``): the field-name
constants (:49-68), the ``get_*_varname`` helpers (:90-138) and ``StationSerialDataDb`` (:547-666) –
structured station array ``stns`` (masked values -> NaN, :159-164), ``stn_ids``, ``days``, ``mth_idx``,
``stn_idxs`` and ``load_obs``.  Station ingest / netCDF I/O stay on the reference path (north_star), so
the container here is built from in-memory arrays or an ``.npz`` file; a netCDF file is accepted only
when the ``netCDF4`` module is importable.
"""
from datetime import datetime, timedelta

import numpy as np

DATE, YMD, YEAR, MONTH, DAY, YDAY = "DATE", "YMD", "YEAR", "MONTH", "DAY", "YDAY"
LON, LAT, ELEV = "longitude", "latitude", "elevation"
STN_ID, STN_NAME, STATE = "station_id", "station_name", "state"
NORM_OBS, TDI, LST = "norm", "tdi", "lst"
OPTIM_NNGH, OPTIM_NNGH_ANOM = "optim_nnghs", "optim_nnghs_anom"
MASK, BAD, CLIMDIV, NORM = "mask", "bad", "climdiv", "norm"
VARIO_NUG, VARIO_PSILL, VARIO_RNG = "vario_nug", "vario_psill", "vario_rng"


def get_lst_varname(mth):
    return LST if mth is None else "lst%02d" % mth


def get_norm_varname(mth):
    return NORM_OBS if mth is None else "norm%02d" % mth


def get_optim_varname(mth):
    return OPTIM_NNGH if mth is None else "optim_nnghs%02d" % mth


def get_optim_anom_varname(mth):
    return OPTIM_NNGH_ANOM if mth is None else "optim_nnghs_anom%02d" % mth


def get_krigparam_varname(mth, krigParam):
    return krigParam if mth is None else "".join([krigParam, "%02d" % mth])


def get_days_metadata(srt_date, end_date):
    """``twx/utils/util_dates.py:117-128``: one record per day with DATE/YEAR/MONTH/DAY/YDAY/YMD."""
    n = (end_date - srt_date).days + 1
    dates = np.array([srt_date + timedelta(days=i) for i in range(n)])
    return get_days_metadata_dates(dates)


def get_days_metadata_dates(dates):
    """``twx/utils/util_dates.py:150-159``."""
    days = np.recarray(dates.size, dtype=[(DATE, np.object_), (YEAR, np.int32), (MONTH, np.int32),
                                          (DAY, np.int32), (YDAY, np.int32), (YMD, np.int32)])
    days[DATE] = dates
    days[YEAR] = [d.year for d in dates]
    days[MONTH] = [d.month for d in dates]
    days[DAY] = [d.day for d in dates]
    days[YDAY] = [d.timetuple().tm_yday for d in dates]
    days[YMD] = [d.year * 10000 + d.month * 100 + d.day for d in dates]
    return days


def month_runs(days):
    """Month groups of a days table (new): maximal runs of consecutive days with one (YEAR, MONTH), as
    twxi_tile_days_mth averages them.  Returns int64 arrays start, ndays, year, month (one entry per run, chronological)."""
    y, m = np.asarray(days[YEAR]), np.asarray(days[MONTH])
    start = np.concatenate([[0], np.flatnonzero((y[1:] != y[:-1]) | (m[1:] != m[:-1])) + 1]).astype(np.int64)
    ndays = np.diff(np.append(start, y.size))
    return start, ndays, y[start].astype(np.int64), m[start].astype(np.int64)


def station_dtype(id_len=16):
    """dtype of the structured station array the hot path reads (numeric fields float64,
    ``station_data.py:159-164``)."""
    dt = [(STN_ID, "U%d" % id_len), (STN_NAME, "U%d" % id_len), (STATE, "U2"),
          (LON, np.float64), (LAT, np.float64), (ELEV, np.float64), (TDI, np.float64),
          (MASK, np.float64), (BAD, np.float64), (CLIMDIV, np.float64)]
    for fn in (get_norm_varname, get_lst_varname, get_optim_varname, get_optim_anom_varname):
        dt += [(fn(m), np.float64) for m in range(1, 13)]
    for p in (VARIO_NUG, VARIO_PSILL, VARIO_RNG):
        dt += [(get_krigparam_varname(m, p), np.float64) for m in range(1, 13)]
    return np.dtype(dt)


class StationSerialDataDb(object):
    """In-memory equivalent of ``twx.db.StationSerialDataDb`` (``station_data.py:547-666``).

    ``source`` is either a path to an ``.npz`` written by :meth:`save` (keys ``stns``, ``obs``,
    ``dates`` as YYYYMMDD int32), a netCDF path (needs ``netCDF4``), or a tuple ``(stns, obs, days)``.
    ``obs`` is float32 ``[ndays, nstns]`` in station (= station-id, ``create_db_all_stations.py:509-515``) order."""

    def __init__(self, source, var_name, vcc_size=None, vcc_nelems=None, vcc_preemption=None, mode="r"):
        if isinstance(source, tuple):
            stns, obs, days = source
        elif str(source).endswith(".npz"):
            with np.load(source, allow_pickle=False) as f:
                stns, obs, ymd = f["stns"], f["obs"], f["dates"]
            dates = np.array([datetime(int(v) // 10000, int(v) // 100 % 100, int(v) % 100) for v in ymd])
            days = get_days_metadata_dates(dates)
        else:
            stns, obs, days = _read_netcdf(source, var_name)
        self.var_name = var_name
        self.stns = stns
        self.stn_ids = np.array(stns[STN_ID])
        if np.any(self.stn_ids[1:] < self.stn_ids[:-1]):
            raise ValueError("station ids must be sorted (DB order is station-id order)")
        self.days = days
        self.var = np.ascontiguousarray(obs, dtype=np.float32)
        if self.var.shape != (days.size, stns.size):
            raise ValueError("obs must be [ndays, nstns]")
        self.mth_idx = {m: np.nonzero(days[MONTH] == m)[0] for m in range(1, 13)}
        self.mth_idx[None] = np.arange(days.size)
        self.stn_idxs = {sid: x for x, sid in enumerate(self.stn_ids)}

    def load_obs(self, stn_ids, mth=None):
        """``station_data.py:619-666``: columns in DB order; 1-D for a single station."""
        if isinstance(stn_ids, np.ndarray):
            num_stns = stn_ids.size
            mask = np.nonzero(np.isin(self.stn_ids, stn_ids))[0]
            obs = self.var[:, mask]
        else:
            num_stns = 1
            obs = self.var[:, self.stn_idxs[stn_ids]]
        if mth is not None:
            obs = np.take(obs, self.mth_idx[mth], axis=0)
        if num_stns == 1:
            obs = obs.reshape(obs.shape[0])
        return obs

    def save(self, path):
        np.savez(path, stns=self.stns, obs=self.var, dates=np.asarray(self.days[YMD], dtype=np.int32))


def _read_netcdf(path, var_name):
    try:
        import netCDF4  # noqa: F401
    except ImportError:
        raise ImportError("netCDF4 is not installed: netCDF station databases stay on the reference "
                          "path; pass (stns, obs, days) arrays or an .npz file instead")
    from netCDF4 import Dataset, num2date, chartostring
    ds = Dataset(path)
    t = ds.variables["time"]
    days = get_days_metadata_dates(np.array(num2date(t[:], t.units)))
    n = len(ds.dimensions[STN_ID])
    names = [v for v in ds.variables if ds.variables[v].dimensions == (STN_ID,)]
    vid = ds.variables[STN_ID]
    ids = chartostring(vid[:]) if len(vid.dimensions) == 2 else vid[:].astype(str)
    dt = [(STN_ID, ids.dtype)] + [(str(v), np.float64) for v in names if v != STN_ID
                                  and ds.variables[v].dtype.kind in "fiu"]
    stns = np.empty(n, dtype=dt)
    stns[STN_ID] = ids
    for v, _ in dt[1:]:
        a = ds.variables[v][:]
        stns[v] = np.ma.filled(np.ma.asarray(a, dtype=np.float64), np.nan)
    obs = np.asarray(ds.variables[var_name][:], dtype=np.float32)
    ds.close()
    return stns, obs, days

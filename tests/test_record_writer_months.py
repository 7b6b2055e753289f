"""TileWriter.open_tile_stream_mthly (CPU): a monthly tile written window by window through the scipy netCDF-3 backend
reads back its arrays, its fill values and the time / time_bnds of every month run, partial months at the record's ends
included."""
import os
from datetime import datetime

import numpy as np


def test_monthly_tile_written_window_by_window(tmp_path):
    from scipy.io import netcdf_file
    from topowx_b200 import synth, db
    from topowx_b200.interp import tiling
    from topowx_b200.interp.tiling import Tiler, TileWriter
    ny, nx = 20, 30
    mask = np.ones((ny, nx), dtype=bool)
    lats, lons = synth.grid_lats(np.arange(ny)), synth.grid_lons(np.arange(nx))
    info = Tiler(dict(mask=mask, lon=lons, lat=lats), [], 10, 10, 5, 5).build_tile_grid_info()
    days = synth.make_days(1979, 2)
    i0, i1 = int(np.flatnonzero(days["YMD"] == 19790110)[0]), int(np.flatnonzero(days["YMD"] == 19800220)[0])
    days = days[i0:i1 + 1]                                            # 1979-01-10 .. 1980-02-20
    start, ndays, year, month = db.month_runs(days)
    nm = start.size
    assert nm == 14 and ndays[0] == 22 and ndays[-1] == 20 and ndays[-2] == 31 and (year[-1], month[-1]) == (1980, 2)
    rng = np.random.default_rng(6)
    vals = rng.normal(10.0, 8.0, (nm, 10, 10)).astype(np.float32)
    vals[:, 2, 3] = tiling.FILL_F4                                    # a failed cell
    tid = info.get_tile_id(1)
    tw = TileWriter(info, str(tmp_path))
    tw._nc = tiling._NcBackend.__new__(tiling._NcBackend)             # the scipy netCDF-3 backend even with netCDF4 around
    tw._nc.nc4, tw._nc.nc3 = None, netcdf_file
    s = tw.open_tile_stream_mthly(tid, "tmax", days)
    for a, b in ((0, 0), (0, 1), (1, 5), (5, 5), (5, 13), (13, 14)):  # windows completing 0, 1, several months
        s.write_months(a, vals[a:b])
    s.close()
    fpath = os.path.join(str(tmp_path), tid, "%s_tmax_mthly.nc" % tid)
    assert os.path.exists(fpath) and not os.path.exists(os.path.join(str(tmp_path), tid, "%s_tmax.nc" % tid))
    ds = netcdf_file(fpath, "r", mmap=False, maskandscale=False)
    v = ds.variables["tmax"]
    got = np.array(v.data).astype(np.float32)                        # big-endian on disk
    assert v.data.dtype.kind == "f" and v.data.dtype.itemsize == 4 and got.shape == (nm, 10, 10)
    assert np.array_equal(got.view(np.int32), vals.view(np.int32))
    assert np.float32(v._FillValue) == tiling.FILL_F4
    assert v.cell_methods.decode() == "area: mean time: maximum within days time: mean over days"
    assert v.grid_mapping.decode() == "crs" and v.units.decode() == "C"
    t, tb = np.array(ds.variables["time"].data), np.array(ds.variables["time_bnds"].data)
    assert ds.variables["time"].units.decode() == "days since 1979-1-10 0:0:0"
    d0 = datetime(1979, 1, 10)
    first = np.array([(datetime(int(y), int(m), 1) - d0).days for y, m in zip(year, month)], dtype=np.float64)
    first[0] = 0.0                                                    # the record starts on the 10th
    assert np.array_equal(tb[:, 0], first)
    assert np.array_equal(tb[:, 1] - tb[:, 0], ndays.astype(np.float64))
    assert tb[-1, 1] == (datetime(1980, 2, 21) - d0).days              # last day + 1
    assert np.array_equal(t, (tb[:, 0] + tb[:, 1]) / 2)
    ds_lat = np.array(ds.variables["lat"].data)
    r0, c0 = info.tile_rc[tid]
    assert np.array_equal(ds_lat, lats[r0:r0 + 10])
    assert np.array_equal(np.array(ds.variables["lon"].data), lons[c0:c0 + 10])
    assert ds.variables["crs"].grid_mapping_name.decode() == "latitude_longitude"
    ds.close()


def test_month_runs():
    from topowx_b200 import db, synth
    days = synth.make_days(1980, 1)
    start, ndays, year, month = db.month_runs(days)
    assert ndays.tolist() == [31, 29, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31]
    assert start.tolist() == np.concatenate([[0], np.cumsum(ndays)[:-1]]).tolist()
    assert (year == 1980).all() and month.tolist() == list(range(1, 13))
    perm = np.concatenate([np.arange(0, 15), np.arange(31, 60), np.arange(15, 31), np.arange(60, days.size)])
    start, ndays, year, month = db.month_runs(days[perm])               # January in two runs: two entries
    assert month[:4].tolist() == [1, 2, 1, 3] and ndays[:3].tolist() == [15, 29, 16]

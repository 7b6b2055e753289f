"""TileWriter.open_tile_stream (CPU): a tile written window by window equals the whole-tile write_tile, variable for
variable, through the scipy netCDF-3 backend."""
import os

import numpy as np


def test_open_tile_stream_equals_write_tile(tmp_path):
    from scipy.io import netcdf_file
    from topowx_b200 import synth
    from topowx_b200.interp import tiling
    from topowx_b200.interp.tiling import Tiler, TileWriter
    ny, nx = 20, 30
    mask = np.ones((ny, nx), dtype=bool)
    lats, lons = synth.grid_lats(np.arange(ny)), synth.grid_lons(np.arange(nx))
    info = Tiler(dict(mask=mask, lon=lons, lat=lats), [], 10, 10, 5, 5).build_tile_grid_info()
    days = synth.make_days(1979, 3)
    nd = days.size
    rng = np.random.default_rng(5)
    daily = rng.integers(-3000, 3000, (nd, 10, 10)).astype(np.int16)
    daily[:, 2, 3] = -32767                                           # a failed cell
    normals = rng.normal(size=(12, 10, 10)).astype(np.float32)
    se = rng.uniform(size=(12, 10, 10)).astype(np.float32)
    ninv = rng.integers(0, 5, (10, 10)).astype(np.int32)
    tid = info.get_tile_id(2)
    whole = TileWriter(info, str(tmp_path / "whole"))
    whole._nc = tiling._NcBackend.__new__(tiling._NcBackend)          # the scipy netCDF-3 backend even with netCDF4 around
    whole._nc.nc4, whole._nc.nc3 = None, netcdf_file
    whole.write_tile(tid, "tmin", days, daily, normals, se, ninv)
    win = TileWriter(info, str(tmp_path / "win"))
    win._nc = whole._nc
    s = win.open_tile_stream(tid, "tmin", days)
    yrs = days["YEAR"]
    bounds = [0, 1, 40] + [int(np.searchsorted(yrs, y)) for y in np.unique(yrs)[1:]] + [nd - 10, nd]
    for a, b in zip(bounds[:-1], bounds[1:]):                         # 1-day, partial and calendar-year windows
        s.write_days(a, daily[a:b])
    s.close(normals, se, ninv)

    def load(root):
        ds = netcdf_file(os.path.join(str(tmp_path / root), tid, "%s_tmin.nc" % tid), "r", mmap=False, maskandscale=False)
        v = {k: (np.array(x.data), {a: getattr(x, a) for a in x._attributes}) for k, x in ds.variables.items()}
        attrs = dict(ds._attributes)
        ds.close()
        return v, attrs
    va, aa = load("whole")
    vb, ab = load("win")
    assert aa == ab and sorted(va) == sorted(vb)
    for k in va:
        assert va[k][0].dtype == vb[k][0].dtype and np.array_equal(va[k][0], vb[k][0]), k
        assert str(va[k][1]) == str(vb[k][1]), k
    assert np.array_equal(vb["tmin"][0], daily)

'''
Tiling of the interpolation grid: the `Tiler` / `TileGridInfo` / `TileWriter` interfaces of
twx/interp/tiling.py:44-537.  `Tiler` works on in-memory arrays (anything indexable like the reference's
netCDF4 variables); `partition_chunks` is the multi-GPU replacement for step25's coordinator rank; `TileWriter` writes
the reference's netCDF tiles (netCDF4 when installed, netCDF-3 through scipy otherwise), `AsyncTileWriter` is the writer
rank as a background thread pool.
'''

__all__ = ['Tiler', 'TileGridInfo', 'TileWriter', 'AsyncTileWriter', 'partition_chunks']

import os
from datetime import datetime

import numpy as np

from ..db import month_runs


class Tiler():
    '''
    Breaks an interpolation grid into tiles and work chunks (tiling.py:44-275).
    '''

    def __init__(self, ds_mask, ds_attr_ls, tile_size_y, tile_size_x, chk_size_y, chk_size_x, path_out=None,
                 process_tiles=False):
        '''
        ds_mask : mapping with 'mask' (2-D), 'lon' (1-D), 'lat' (1-D, descending) – a netCDF4.Dataset's
            `.variables` or a dict of arrays.
        ds_attr_ls : list of (name, 2-D array-like) auxiliary predictor grids, in work-chunk plane order.
        '''
        v = ds_mask.variables if hasattr(ds_mask, 'variables') else ds_mask
        self.mask = np.array(v['mask'][:], dtype=bool)
        self.lons = np.asarray(v['lon'][:])
        self.lats = np.asarray(v['lat'][:])
        self.nrows = self.lats.size
        self.ncols = self.lons.size
        if self.nrows % tile_size_y or self.ncols % tile_size_x:
            raise ValueError("the grid size must be evenly divisible by the tile size")
        if tile_size_y % chk_size_y or tile_size_x % chk_size_x:
            raise ValueError("the tile size must be evenly divisible by the chunk size")
        self.tile_size_y = tile_size_y
        self.tile_size_x = tile_size_x
        self.chk_size_y = chk_size_y
        self.chk_size_x = chk_size_x
        self.attrs = []
        for varname, ds in ds_attr_ls:
            attr = ds.variables[varname] if hasattr(ds, 'variables') else ds
            if hasattr(attr, 'set_auto_maskandscale'):
                attr.set_auto_maskandscale(False)
            self.attrs.append(attr)
        self.tile_ids, self.tile_rc = self.__build_tile_dicts(self.nrows, self.ncols, tile_size_y, tile_size_x, self.mask)
        self.chk_size_i = 5 + len(self.attrs)
        self.wrk_chk = np.zeros((self.chk_size_i, chk_size_y, chk_size_x)) * np.nan
        try:
            self.process_tiles = list(process_tiles)
        except TypeError:
            if type(process_tiles) == bool and process_tiles:
                self.process_tiles = self.get_incomplete_tile_nums(path_out)
            else:
                self.process_tiles = None
        self.__set_tile_chks()

    def __set_tile_chks(self):
        k = 0
        self.tile_chks = []
        self.ntiles = 0
        for i in np.arange(0, self.nrows, self.tile_size_y):
            for j in np.arange(0, self.ncols, self.tile_size_x):
                msk_tile = self.mask[i:i + self.tile_size_y, j:j + self.tile_size_x]
                if msk_tile.any():
                    process_tile = self.process_tiles is None or k in self.process_tiles
                    if process_tile:
                        for y in np.arange(0, self.tile_size_y, self.chk_size_y):
                            for x in np.arange(0, self.tile_size_x, self.chk_size_x):
                                self.tile_chks.append((k, int(i), int(j), int(y), int(x)))
                        self.ntiles += 1
                    k += 1
        self.iter_x = 0
        self.ntile_chks = len(self.tile_chks)

    def build_chunk(self, chk, out=None):
        '''The work chunk f8[(5+N), Y, X] of entry `chk` = (k, i, j, y, x) of tile_chks (tiling.py:179-215).'''
        k, i, j, y, x = chk
        w = self.wrk_chk if out is None else out
        cy, cx = self.chk_size_y, self.chk_size_x
        rcgrid = np.mgrid[y:y + cy, x:x + cx]
        w[0, :, :] = rcgrid[0, :, :]
        w[1, :, :] = rcgrid[1, :, :]
        w[2, :, :] = self.mask[i + y:i + y + cy, j + x:j + x + cx]
        w[3, :, :] = self.lats[i + y:i + y + cy][:, None]
        w[4, :, :] = self.lons[j + x:j + x + cx][None, :]
        for z, attr in enumerate(self.attrs):
            w[5 + z, :, :] = attr[i + y:i + y + cy, j + x:j + x + cx]
        return k, w

    def next(self):
        '''
        Next work chunk: (tile number, wrk_chk f8[(5+N), Y, X]); planes 0 row, 1 col, 2 mask, 3 lat, 4 lon,
        then the N predictors.  Raises StopIteration at the end (tiling.py:167-217).
        '''
        if self.iter_x == self.ntile_chks:
            raise StopIteration()
        k, w = self.build_chunk(self.tile_chks[self.iter_x])
        self.iter_x += 1
        return k, w

    __next__ = next

    def __iter__(self):
        return self

    def __build_tile_dicts(self, nrows, ncols, tile_size_y, tile_size_x, mask):
        tile_ids = {}
        tile_info = {}
        x = 0
        cnt_y = 0
        for i in np.arange(0, nrows, tile_size_y):
            cnt_x = 0
            for j in np.arange(0, ncols, tile_size_x):
                if mask[i:i + tile_size_y, j:j + tile_size_x].any():
                    atileid = "".join(["h%02d" % (cnt_x,), "v%02d" % (cnt_y,)])
                    tile_ids[x] = atileid
                    tile_info[atileid] = (int(i), int(j))
                    x += 1
                cnt_x += 1
            cnt_y += 1
        return tile_ids, tile_info

    def build_tile_grid_info(self):
        return TileGridInfo(self.tile_ids, self.tile_rc, self.ntiles, self.lons, self.lats, self.tile_size_y,
                            self.tile_size_x, self.chk_size_y, self.chk_size_x, self.chk_size_i)

    def get_incomplete_tile_nums(self, path_out):
        name_to_id = {a_name: a_id for a_id, a_name in self.tile_ids.items()}
        all_ids = np.unique(list(self.tile_ids.keys()))
        names_done = [n for n in os.listdir(path_out) if n in name_to_id]
        ids_done = np.unique([name_to_id[a_name] for a_name in names_done])
        return all_ids[~np.isin(all_ids, ids_done)]


class TileGridInfo():
    '''Information on tiles and work chunks of an interpolation grid (tiling.py:277-302).'''

    def __init__(self, tile_ids, tile_rc, ntiles, lons, lats, tile_size_y, tile_size_x, chk_size_y, chk_size_x,
                 chk_size_i):
        self.tile_ids = tile_ids
        self.tile_rc = tile_rc
        self.ntiles = ntiles
        self.lons = lons
        self.lats = lats
        self.tile_size_y = tile_size_y
        self.tile_size_x = tile_size_x
        self.chk_size_y = chk_size_y
        self.chk_size_x = chk_size_x
        self.chk_size_i = chk_size_i
        self.chks_per_tile = (tile_size_x // chk_size_x) * (tile_size_y // chk_size_y)
        self.nchks = self.chks_per_tile * ntiles

    def get_tile_id(self, tile_num):
        return self.tile_ids[tile_num]


def partition_chunks(tile_chks, mask, tile_size_y, tile_size_x, world_size, rank=None):
    '''
    Static multi-GPU partition of the ordered chunk list (replaces the coordinator rank's first-come dispatch,
    step25_mpi_interp_tair.py:293-305): whole tiles are assigned to ranks by greedy longest-processing-time on
    the number of unmasked cells, chunks keep their reference order inside a rank.  Deterministic, so every rank
    computes the same partition without communication.  Returns the per-rank lists, or rank's list.
    '''
    tiles = {}
    for c in tile_chks:
        tiles.setdefault(c[0], []).append(c)
    work = []
    for k, chks in tiles.items():
        _, i, j, _, _ = chks[0]
        work.append((int(mask[i:i + tile_size_y, j:j + tile_size_x].sum()), k))
    work.sort(key=lambda t: (-t[0], t[1]))
    loads = [0] * world_size
    owner = {}
    for n, k in work:
        r = min(range(world_size), key=lambda q: (loads[q], q))
        owner[k] = r
        loads[r] += n
    parts = [[c for c in tile_chks if owner[c[0]] == r] for r in range(world_size)]
    return parts if rank is None else parts[rank]


SCALE_FACTOR = np.float32(0.01)                      # tiling.py:36
FILL_I2, FILL_I4 = -32767, -2147483647               # netCDF4.default_fillvals
FILL_F4 = np.float32(9.969209968386869e+36)
# long name, units, standard name, missing value, cell method (tiling.py:38-42)
VAR_ATTRS = {'tmin': ("minimum air temperature", "C", "air_temperature", FILL_I2, "minimum"),
             'tmax': ("maximum air temperature", "C", "air_temperature", FILL_I2, "maximum")}


def _date2num(dates, d0):
    """days since d0 (netCDF4.date2num with units 'days since Y-M-D 0:0:0', calendar standard)."""
    return np.array([(datetime(d.year, d.month, d.day) - d0).total_seconds() / 86400.0 for d in dates])


class _NcBackend(object):
    """The handful of netCDF calls TileWriter needs, over netCDF4 when it imports and over scipy.io.netcdf_file
    (netCDF-3, 64-bit offsets: no chunking, no compression; same dimensions, variables, attributes and fill values)
    otherwise."""

    def __init__(self):
        try:
            import netCDF4
            self.nc4 = netCDF4
        except ImportError:
            self.nc4 = None
            from scipy.io import netcdf_file
            self.nc3 = netcdf_file

    def open(self, fpath, mode):
        if self.nc4 is not None:
            return self.nc4.Dataset(fpath, mode if mode != 'a' else 'r+')
        return self.nc3(fpath, mode, mmap=False, version=2)

    def create_variable(self, ds, name, dtype, dims, fill_value=None, chunksizes=None):
        if self.nc4 is not None:
            return ds.createVariable(name, dtype, dims, fill_value=fill_value if fill_value is not None else False,
                                     chunksizes=chunksizes)
        v = ds.createVariable(name, np.dtype(dtype), dims)
        if fill_value is not None:
            v._FillValue = np.array(fill_value, dtype=np.dtype(dtype))
            if dims:
                v[:] = fill_value                              # netCDF-3 has no default fill on unwritten data
        return v


class TileWriter():
    '''
    A utility class for writing out interpolation results to netCDF tiles (tiling.py:304-537): one file
    <path_out>/<tile_id>/<tile_id>_<varname>.nc per tile and variable with the int16 daily values (scale_factor 0.01),
    the float32 1981-2010 normals and their kriging standard errors and the int32 count of Tmin >= Tmax days, CF-1.6
    attributes and the fill values of netCDF4.default_fillvals.  Written with netCDF4 when that module imports (then with
    the reference's chunk sizes), otherwise as netCDF-3 (64-bit offset) through scipy.io.netcdf_file.
    `write_tile` (new) writes a whole tile at once: the GPU path produces whole tiles.
    '''

    def __init__(self, tile_grid_info, path_out):
        self.tile_ids = tile_grid_info.tile_ids
        self.tile_rc = tile_grid_info.tile_rc
        self.ntiles = tile_grid_info.ntiles
        self.lons = tile_grid_info.lons
        self.lats = tile_grid_info.lats
        self.path_out = path_out
        self.tile_size_y = tile_grid_info.tile_size_y
        self.tile_size_x = tile_grid_info.tile_size_x
        self.chk_size_y = tile_grid_info.chk_size_y
        self.chk_size_x = tile_grid_info.chk_size_x
        self._nc = _NcBackend()
        self.format = "netCDF4" if self._nc.nc4 is not None else "netCDF3_64bit (scipy.io.netcdf_file)"

    def _fpath(self, tile_id, varname):
        return os.path.join(self.path_out, tile_id, "%s_%s.nc" % (tile_id, varname))

    def _open_dataset(self, tile_id, varname, days):
        fpath = self._fpath(tile_id, varname)
        if os.path.exists(fpath):
            return self._nc.open(fpath, 'a')
        os.makedirs(os.path.join(self.path_out, tile_id), exist_ok=True)
        return self._create_ncdf(fpath, tile_id, varname, days)

    def _new_tile_dataset(self, fpath, tile_id, days, ntime, title, comment, extra_dims=()):
        """A new tile file with the global attributes, the dimensions time (ntime), lat, lon, nv and extra_dims, and the
        time coordinate (values left to the caller) in days since the record's first day.  Returns (ds, d0, units)."""
        from .. import __version__ as twx_version
        nc = self._nc
        ds = nc.open(fpath, 'w')
        ds.title = "".join([title, str(days['YMD'][0]), "-", str(days['YMD'][-1])])
        ds.institution = "University of Montana"
        ds.source = "TopoWx %s (topowx_b200 GPU path)" % twx_version
        ds.history = "".join(["Created on: ", datetime.strftime(datetime.today(), "%Y-%m-%d")])
        ds.references = "http://www.ntsg.umt.edu/project/TopoWx"
        ds.comment = comment
        ds.Conventions = "CF-1.6"
        ds.createDimension('time', ntime)
        str_row, str_col = self.tile_rc[tile_id]
        ds.createDimension('lat', self.lats[str_row:str_row + self.tile_size_y].size)
        ds.createDimension('lon', self.lons[str_col:str_col + self.tile_size_x].size)
        ds.createDimension('nv', 2)
        for name, size in extra_dims:
            ds.createDimension(name, size)
        min_date = days['DATE'][0]
        d0 = datetime(min_date.year, min_date.month, min_date.day)
        units = "".join(["days since ", str(min_date.year), "-", str(min_date.month), "-", str(min_date.day), " 0:0:0"])
        times = nc.create_variable(ds, 'time', 'f8', ('time',))
        times.long_name = "time"
        times.units = units
        times.standard_name = "time"
        times.calendar = "standard"
        times.bounds = 'time_bnds'
        nc.create_variable(ds, 'time_bnds', 'f8', ('time', 'nv'))
        return ds, d0, units

    def _add_grid(self, ds, tile_id):
        """lat, lon and the crs grid mapping of the tile."""
        nc = self._nc
        str_row, str_col = self.tile_rc[tile_id]
        latitudes = nc.create_variable(ds, 'lat', 'f8', ('lat',))
        latitudes.long_name = "latitude"
        latitudes.units = "degrees_north"
        latitudes.standard_name = "latitude"
        latitudes[:] = self.lats[str_row:str_row + self.tile_size_y]
        longitudes = nc.create_variable(ds, 'lon', 'f8', ('lon',))
        longitudes.long_name = "longitude"
        longitudes.units = "degrees_east"
        longitudes.standard_name = "longitude"
        longitudes[:] = self.lons[str_col:str_col + self.tile_size_x]
        crs = nc.create_variable(ds, 'crs', 'i2', ())
        crs.grid_mapping_name = "latitude_longitude"
        crs.longitude_of_prime_meridian = 0.0
        crs.semi_major_axis = 6378137.0
        crs.inverse_flattening = 298.257223563

    def _create_ncdf(self, fpath, tile_id, varname, days):
        nc = self._nc
        ds, d0, units = self._new_tile_dataset(fpath, tile_id, days, days.size, "Daily Interpolated Meteorological Data ",
                                               "30-arcsec spatial resolution, daily timestep", [('time_normals', 12)])
        time_nums = _date2num(days['DATE'], d0) + 0.5
        ds.variables['time'][:] = time_nums
        ds.variables['time_bnds'][:] = np.stack([time_nums - 0.5, time_nums + 0.5], axis=1)
        time_means = nc.create_variable(ds, 'time_normals', 'f8', ('time_normals',))
        time_means.long_name = "time"
        time_means.units = units
        time_means.standard_name = "time"
        time_means.calendar = "standard"
        time_means.climatology = "climatology_bounds"
        time_means.comment = "Time dimension for the 1981-2010 monthly normals"
        clim_bnds = nc.create_variable(ds, 'climatology_bounds', 'f8', ('time_normals', 'nv'))
        tm, cb = np.empty(12), np.empty((12, 2))
        for mth in range(1, 13):
            mth_next = mth + 1 if mth != 12 else 1
            a, b = datetime(1981, mth, 1), datetime(1981 if mth != 12 else 1982, mth_next, 1)
            mid = a + (b - a) / 2
            tm[mth - 1] = _date2num([datetime(mid.year, mid.month, mid.day)], d0)[0]
            cb[mth - 1] = _date2num([datetime(1981, mth, 1), datetime(2010 if mth != 12 else 2011, mth_next, 1)], d0)
        time_means[:] = tm
        clim_bnds[:] = cb
        self._add_grid(ds, tile_id)
        self._add_dim_vars(ds, varname, days)
        return ds

    def _add_dim_vars(self, ds, varname, days):
        nc = self._nc
        long_name, units, standard_name, fill_value, cell_method = VAR_ATTRS[varname]

        def grid_mapping(v):
            v.coordinates = "lat lon"
            v.grid_mapping = "crs"
        mainvar = nc.create_variable(ds, varname, 'i2', ('time', 'lat', 'lon'), fill_value=fill_value,
                                     chunksizes=(days.size, self.chk_size_y, self.chk_size_x))
        mainvar.long_name = long_name
        mainvar.units = units
        mainvar.standard_name = standard_name
        mainvar.scale_factor = SCALE_FACTOR
        mainvar.cell_methods = "".join(["area: mean ", "time: ", cell_method])
        grid_mapping(mainvar)
        avar = nc.create_variable(ds, varname + "_normal", 'f4', ('time_normals', 'lat', 'lon'), fill_value=FILL_F4,
                                  chunksizes=(12, self.chk_size_y, self.chk_size_x))
        avar.long_name = "normal " + long_name
        avar.units = units
        avar.standard_name = standard_name
        avar.ancillary_variables = varname + "_se"
        avar.comment = "The 1981-2010 monthly normals"
        avar.cell_methods = "time: %s within years time: mean over years" % cell_method
        grid_mapping(avar)
        avar = nc.create_variable(ds, varname + "_se", 'f4', ('time_normals', 'lat', 'lon'), fill_value=FILL_F4,
                                  chunksizes=(12, self.chk_size_y, self.chk_size_x))
        avar.long_name = long_name + " kriging standard error"
        avar.standard_name = 'air_temperature standard_error'
        avar.units = units
        avar.comment = "The uncertainty in the 1981-2010 monthly normals"
        grid_mapping(avar)
        avar = nc.create_variable(ds, "inconsist_tair", 'i4', ('lat', 'lon'), fill_value=FILL_I4,
                                  chunksizes=(self.chk_size_y, self.chk_size_x))
        avar.long_name = "number of days interpolated tmin >= tmax"
        avar.units = "days"
        avar.comment = ("The number of days daily tmin/tmax had to be adjusted due to interpolated tmin being >= "
                        "interpolated tmax")
        grid_mapping(avar)

    def _write(self, ds, varname, sl_r, sl_c, daily_vals, mthly_normals, mthly_normals_se, ninvalid):
        v = ds.variables[varname]
        if hasattr(v, 'set_auto_maskandscale'):
            v.set_auto_maskandscale(False)                     # data is already scaled int16 (tiling.py:529)
        v[:, sl_r, sl_c] = daily_vals
        ds.variables[varname + "_normal"][:, sl_r, sl_c] = mthly_normals
        ds.variables[varname + "_se"][:, sl_r, sl_c] = mthly_normals_se
        ds.variables['inconsist_tair'][sl_r, sl_c] = ninvalid
        ds.close()

    def write_tile_chunk(self, tile_id, varname, days, str_row, str_col, daily_vals, mthly_normals, mthly_normals_se,
                         ninvalid):
        '''
        Writes out a work chunk for a netCDF tile; the file is created on first use (tiling.py:488-537).
        daily_vals int16 [N, chk_y, chk_x] (already scaled), mthly_normals / mthly_normals_se [12, chk_y, chk_x],
        ninvalid int [chk_y, chk_x]; str_row / str_col = origin of the chunk inside the tile.
        '''
        ds = self._open_dataset(tile_id, varname, days)
        self._write(ds, varname, slice(str_row, str_row + self.chk_size_y), slice(str_col, str_col + self.chk_size_x),
                    daily_vals, mthly_normals, mthly_normals_se, ninvalid)

    def write_tile(self, tile_id, varname, days, daily_vals, mthly_normals, mthly_normals_se, ninvalid):
        '''New: a whole tile [N, tile_y, tile_x] in one call (one file creation, one pass over the data).'''
        fpath = self._fpath(tile_id, varname)
        if os.path.exists(fpath):
            os.remove(fpath)
        ds = self._open_dataset(tile_id, varname, days)
        self._write(ds, varname, slice(None), slice(None), daily_vals, mthly_normals, mthly_normals_se, ninvalid)

    def open_tile_stream(self, tile_id, varname, days):
        '''
        New: a whole tile written window by window (PtInterpTair.interp_chunk_stream).  Returns a handle with
        `write_days(day0, vals)` (int16 [n, tile_y, tile_x] for days day0 .. day0+n-1) and `close(normals, se, ninvalid)`.
        One dataset stays open from the first window to close, so no window is read back or rewritten; the file equals what
        write_tile writes from the whole-record result.  The scipy netCDF-3 backend holds a variable in host memory until
        close (the whole record of the tile), netCDF4 writes each window through.
        '''
        fpath = self._fpath(tile_id, varname)
        if os.path.exists(fpath):
            os.remove(fpath)
        return _TileStream(self._open_dataset(tile_id, varname, days), varname)

    def _fpath_mthly(self, tile_id, varname):
        return os.path.join(self.path_out, tile_id, "%s_%s_mthly.nc" % (tile_id, varname))

    def open_tile_stream_mthly(self, tile_id, varname, days):
        '''
        New: the monthly means of a tile (PtInterpTair.interp_chunk_stream(months=True)) written as the windows complete
        them, to <tile_id>_<varname>_mthly.nc beside the daily file.  One time step per month run of `days`
        (db.month_runs): `time` is its middle, `time_bnds` its first day and its last day + 1 in the record, so a month the
        record covers in part is bounded by the days it has.  Returns a handle with `write_months(m0, vals)` (float32
        [n, tile_y, tile_x] for months m0 .. m0+n-1) and `close()`.
        '''
        nc = self._nc
        fpath = self._fpath_mthly(tile_id, varname)
        if os.path.exists(fpath):
            os.remove(fpath)
        os.makedirs(os.path.join(self.path_out, tile_id), exist_ok=True)
        start, ndays, _, _ = month_runs(days)
        ds, d0, _ = self._new_tile_dataset(fpath, tile_id, days, start.size, "Monthly Interpolated Meteorological Data ",
                                           "30-arcsec spatial resolution, monthly timestep")
        first = _date2num(days['DATE'][start], d0)
        last1 = _date2num(days['DATE'][start + ndays - 1], d0) + 1.0
        ds.variables['time'][:] = (first + last1) / 2.0
        ds.variables['time_bnds'][:] = np.stack([first, last1], axis=1)
        self._add_grid(ds, tile_id)
        long_name, units, standard_name, _, cell_method = VAR_ATTRS[varname]
        v = nc.create_variable(ds, varname, 'f4', ('time', 'lat', 'lon'), fill_value=FILL_F4,
                               chunksizes=(1, self.chk_size_y, self.chk_size_x))
        v.long_name = "monthly mean " + long_name
        v.units = units
        v.standard_name = standard_name
        v.cell_methods = "area: mean time: %s within days time: mean over days" % cell_method
        v.comment = ("Mean of the month's daily values as stored in the daily tile (int16, scale_factor 0.01); a month the "
                     "record covers in part is the mean of the days it has")
        v.coordinates = "lat lon"
        v.grid_mapping = "crs"
        return _MonthStream(ds, varname)


class _TileStream(object):
    '''Open dataset of TileWriter.open_tile_stream.'''

    def __init__(self, ds, varname):
        self.ds = ds
        self.varname = varname
        self.v = ds.variables[varname]
        if hasattr(self.v, 'set_auto_maskandscale'):
            self.v.set_auto_maskandscale(False)                # data is already scaled int16 (tiling.py:529)

    def write_days(self, day0, vals):
        self.v[day0:day0 + len(vals), :, :] = vals

    def close(self, mthly_normals, mthly_normals_se, ninvalid):
        ds = self.ds
        ds.variables[self.varname + "_normal"][:, :, :] = mthly_normals
        ds.variables[self.varname + "_se"][:, :, :] = mthly_normals_se
        ds.variables['inconsist_tair'][:, :] = ninvalid
        ds.close()


class _MonthStream(object):
    '''Open dataset of TileWriter.open_tile_stream_mthly.'''

    def __init__(self, ds, varname):
        self.ds = ds
        self.v = ds.variables[varname]

    def write_months(self, m0, vals):
        if len(vals):
            self.v[m0:m0 + len(vals), :, :] = vals

    def close(self):
        self.ds.close()


class AsyncTileWriter(object):
    '''
    New: the writer rank of step25 (step25:200-264: workers send finished chunks, one rank writes) as a background thread
    pool fed by the GPU loop.  `submit(tile_id, out)` takes the result dict of PtInterpTair.interp_chunk for a whole tile
    (the arrays are copied first unless copy=False, so pinned staging buffers can be reused at once) and writes both
    variables; `fmt` = 'nc' (TileWriter) or 'raw' (one .npy per array: no netCDF dependency, no format overhead).
    '''

    def __init__(self, tile_grid_info, path_out, days, fmt='nc', nthreads=2):
        from concurrent.futures import ThreadPoolExecutor
        self.tw = TileWriter(tile_grid_info, path_out)
        self.path_out = path_out
        self.days = days
        self.fmt = fmt
        self.pool = ThreadPoolExecutor(max_workers=nthreads)
        self.futures = []
        self.bytes_written = 0

    def _job(self, tile_id, o):
        n = 0
        if self.fmt == 'raw':
            d = os.path.join(self.path_out, tile_id)
            os.makedirs(d, exist_ok=True)
            for k, a in o.items():
                if a is not None:
                    np.save(os.path.join(d, "%s_%s.npy" % (tile_id, k)), a)
                    n += a.nbytes
            return n
        for v in ('tmin', 'tmax'):
            self.tw.write_tile(tile_id, v, self.days, o[v], o[v + '_norm'], o[v + '_se'], o['ninvalid'])
            n += os.path.getsize(self.tw._fpath(tile_id, v))
        return n

    def submit(self, tile_id, out, copy=True):
        o = {k: (None if a is None else (np.array(a, copy=True) if copy else np.asarray(a))) for k, a in out.items()}
        self.futures.append(self.pool.submit(self._job, tile_id, o))

    def wait(self):
        for f in self.futures:
            self.bytes_written += f.result()
        self.futures = []
        return self.bytes_written

    def close(self):
        self.wait()
        self.pool.shutdown()

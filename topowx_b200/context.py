"""Python-side handle of one libtwxi context (one temperature variable on one GPU) and thin batch wrappers
around the C-ABI stages.  Host logic only: every number comes from the CUDA library."""
import ctypes as C
import weakref

import numpy as np

from . import _lib
from . import db
from ._lib import lib, check, ptr, Points, MEM_HOST, MEM_DEVICE


def _f8(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _dtype_name(a):
    """'float64', 'int16', ... of a numpy array or a torch tensor."""
    return str(a.dtype).replace("torch.", "")


class TwxiContext(object):
    """Device-resident station table of the stations selected by ``stn_mask`` (default: isnan(bad), as in
    PtInterpTair.__init__, twx/interp/interp_tair.py:481-487), in DB order, plus the observations."""

    def __init__(self, stn_da, stn_mask=None, device=0, with_obs=True):
        stns = stn_da.stns
        self.stn_da = stn_da
        self.mask = np.ones(stns.size, dtype=bool) if stn_mask is None else np.asarray(stn_mask, dtype=bool)
        self.gidx = np.nonzero(self.mask)[0]                  # ctx index -> DB index
        self.stns = stns[self.mask]
        self.n = int(self.gidx.size)
        self.local_of_db = -np.ones(stns.size, dtype=np.int64)
        self.local_of_db[self.gidx] = np.arange(self.n)
        s = self.stns

        def mthly(fn):
            return _f8(np.stack([s[fn(m)] for m in range(1, 13)]))
        vario = lambda p: _f8(np.stack([s[db.get_krigparam_varname(m, p)] for m in range(1, 13)]))
        self._h = C.c_void_p()
        arrs = [_f8(s[db.LON]), _f8(s[db.LAT]), _f8(s[db.ELEV]), _f8(s[db.TDI]),
                mthly(db.get_lst_varname), mthly(db.get_norm_varname), mthly(db.get_optim_varname),
                mthly(db.get_optim_anom_varname), vario(db.VARIO_NUG), vario(db.VARIO_PSILL), vario(db.VARIO_RNG)]
        check(lib.twxi_ctx_create(C.byref(self._h), int(device), self.n, *[ptr(a) for a in arrs]))
        self._finalizer = weakref.finalize(self, lib.twxi_ctx_destroy, self._h)
        self.device = int(device)
        self.ndays = 0
        if with_obs and getattr(stn_da, "var", None) is not None:
            self.set_obs(stn_da)
        # climate divisions known to the DB: keys of _get_rgn_nnghs_dict (interp_tair.py:487-492,594-610)
        dom = self.stns[np.isfinite(self.stns[db.MASK])] if db.MASK in self.stns.dtype.names else self.stns
        if db.CLIMDIV in self.stns.dtype.names:
            cd = dom[db.CLIMDIV]
            self.climdivs = np.unique(cd[np.isfinite(cd)]).astype(np.float64)
            check(lib.twxi_ctx_set_climdivs(self._h, ptr(self.climdivs), int(self.climdivs.size)))

    @property
    def handle(self):
        return self._h

    def set_obs(self, stn_da):
        obs = np.ascontiguousarray(np.asarray(stn_da.var)[:, self.gidx], dtype=np.float32)
        days = stn_da.days
        month = np.ascontiguousarray(days[db.MONTH], dtype=np.int32)
        year = np.ascontiguousarray(days[db.YEAR], dtype=np.int32)
        check(lib.twxi_ctx_set_obs(self._h, ptr(obs), int(obs.shape[0]), ptr(month), ptr(year)))
        self.ndays = int(obs.shape[0])
        self.mth_idx = stn_da.mth_idx

    def set_stream(self, stream_ptr):
        check(lib.twxi_ctx_set_stream(self._h, C.c_void_p(stream_ptr)))

    def close(self):
        self._finalizer()

    # ---- helpers -------------------------------------------------------------------------------------
    def rm_indices(self, stns_rm, npts=1):
        """station ids (str / array of str, StationSelect.__set_pt, station_select.py:74-77) -> ctx indices."""
        if stns_rm is None:
            return None
        if isinstance(stns_rm, str):
            stns_rm = np.array([stns_rm])
        elif not isinstance(stns_rm, np.ndarray):
            raise Exception("stns_rm must be str, unicode, or numpy array of str/unicode")
        loc = [self.local_of_db[self.stn_da.stn_idxs[s]] for s in stns_rm if s in self.stn_da.stn_idxs]
        loc = [int(i) for i in loc if i >= 0]
        if len(loc) > _lib.MAX_RM:
            raise ValueError("at most %d stations can be left out per point" % _lib.MAX_RM)
        if not loc:
            return None
        return np.tile(np.asarray(loc, dtype=np.int32), (npts, 1))

    def _points(self, lat, lon, elev=None, tdi=None, lst=None, rm_idx=None, rm_zero=False):
        lat, lon = _f8(np.atleast_1d(lat)), _f8(np.atleast_1d(lon))
        keep = [lat, lon]
        elev = None if elev is None else _f8(np.atleast_1d(elev))
        tdi = None if tdi is None else _f8(np.atleast_1d(tdi))
        lst = None if lst is None else _f8(np.asarray(lst).reshape(lat.size, 12))
        n_rm = 0
        if rm_idx is not None:
            rm_idx = np.ascontiguousarray(np.asarray(rm_idx, dtype=np.int32).reshape(lat.size, -1))
            n_rm = rm_idx.shape[1]
        keep += [elev, tdi, lst, rm_idx]
        p = Points(int(lat.size), ptr(lat), ptr(lon), ptr(elev), ptr(tdi), ptr(lst), ptr(rm_idx), n_rm, int(bool(rm_zero)))
        return p, keep

    # ---- stages ----------------------------------------------------------------------------------------
    def knn(self, lat, lon, nnghs, rm_idx=None, rm_zero=False):
        lat, lon = _f8(np.atleast_1d(lat)), _f8(np.atleast_1d(lon))
        n, k1 = lat.size, int(nnghs) + 1
        idx = np.empty((n, k1), dtype=np.int32)
        dist = np.empty((n, k1), dtype=np.float64)
        wgt = np.empty((n, k1), dtype=np.float64)
        st = np.empty(n, dtype=np.uint8)
        n_rm = 0
        if rm_idx is not None:
            rm_idx = np.ascontiguousarray(np.asarray(rm_idx, dtype=np.int32).reshape(n, -1))
            n_rm = rm_idx.shape[1]
        check(lib.twxi_knn(self._h, n, ptr(lat), ptr(lon), ptr(rm_idx), n_rm, int(bool(rm_zero)), k1,
                           ptr(idx), ptr(dist), ptr(wgt), ptr(st), MEM_HOST))
        return idx, dist, wgt, st

    def nngh_params(self, lat, lon, rm_idx=None, rm_zero=False):
        p, keep = self._points(lat, lon, rm_idx=rm_idx, rm_zero=rm_zero)
        n = p.npts
        kn, ka = np.empty((n, 12), dtype=np.int32), np.empty((n, 12), dtype=np.int32)
        vario = np.empty((n, 12, 3), dtype=np.float64)
        st = np.empty(n, dtype=np.uint8)
        check(lib.twxi_nngh_params(self._h, C.byref(p), ptr(kn), ptr(ka), ptr(vario), ptr(st), MEM_HOST))
        return kn, ka, vario, st

    def krig(self, lat, lon, elev, lst, mth=0, nnghs=None, vario=None, rm_idx=None, rm_zero=False):
        p, keep = self._points(lat, lon, elev=elev, lst=lst, rm_idx=rm_idx, rm_zero=rm_zero)
        n, nm = p.npts, (1 if mth else 12)
        mean, var = np.empty((n, nm)), np.empty((n, nm))
        st = np.empty(n, dtype=np.uint8)
        nn = None if nnghs is None else np.ascontiguousarray(np.broadcast_to(nnghs, (n,)), dtype=np.int32)
        vo = None if vario is None else _f8(np.broadcast_to(vario, (n, 3)))
        check(lib.twxi_krig(self._h, C.byref(p), int(mth), ptr(nn), ptr(vo), ptr(mean), ptr(var), ptr(st), MEM_HOST))
        return mean, var, st

    def fit_vario(self, lat, lon, mth=0, nnghs=None, rm_idx=None, rm_zero=False):
        """twxi_fit_vario: (nugget, psill, range) [n, 12 or 1, 3] of the neighbourhoods of the points, status [n]."""
        p, keep = self._points(lat, lon, rm_idx=rm_idx, rm_zero=rm_zero)
        n, nm = p.npts, (1 if mth else 12)
        vario = np.empty((n, nm, 3))
        st = np.empty(n, dtype=np.uint8)
        nn = None if nnghs is None else np.ascontiguousarray(np.broadcast_to(nnghs, (n,)), dtype=np.int32)
        check(lib.twxi_fit_vario(self._h, C.byref(p), int(mth), ptr(nn), ptr(vario), ptr(st), MEM_HOST))
        return vario, st

    def krig_all(self, lat, lon, elev, lst, nnghs, rm_idx=None, rm_zero=False):
        """twxi_krig_all: variogram fit + kriging of all 12 months with ``nnghs`` neighbours per point.
        Returns mean, var [n, 12], vario [n, 12, 3], status [n]."""
        p, keep = self._points(lat, lon, elev=elev, lst=lst, rm_idx=rm_idx, rm_zero=rm_zero)
        n = p.npts
        mean, var, vario = np.empty((n, 12)), np.empty((n, 12)), np.empty((n, 12, 3))
        st = np.empty(n, dtype=np.uint8)
        nn = np.ascontiguousarray(np.broadcast_to(nnghs, (n,)), dtype=np.int32)
        check(lib.twxi_krig_all(self._h, C.byref(p), ptr(nn), ptr(mean), ptr(var), ptr(vario), ptr(st), MEM_HOST))
        return mean, var, vario, st

    def gwr_hat(self, lat, lon, elev, tdi, lst, mth, nnghs=None, rm_idx=None, rm_zero=False, kmax=_lib.MAX_NNGHS):
        p, keep = self._points(lat, lon, elev=elev, tdi=tdi, lst=lst, rm_idx=rm_idx, rm_zero=rm_zero)
        n = p.npts
        k = np.zeros(n, dtype=np.int32)
        idx = np.zeros((n, kmax), dtype=np.int32)
        z = np.zeros((n, kmax))
        st = np.empty(n, dtype=np.uint8)
        nn = None if nnghs is None else np.ascontiguousarray(np.broadcast_to(nnghs, (n,)), dtype=np.int32)
        check(lib.twxi_gwr_hat(self._h, C.byref(p), int(mth), ptr(nn), int(kmax), ptr(k), ptr(idx), ptr(z), ptr(st), MEM_HOST))
        return k, idx, z, st

    def gwr_mth(self, lat, lon, elev, tdi, lst, mth, pt_norm, nnghs=None, rm_idx=None, rm_zero=False):
        p, keep = self._points(lat, lon, elev=elev, tdi=tdi, lst=lst, rm_idx=rm_idx, rm_zero=rm_zero)
        n = p.npts
        D = int(self.mth_idx[mth].size)
        out = np.empty((n, D))
        st = np.empty(n, dtype=np.uint8)
        ptn = _f8(np.broadcast_to(pt_norm, (n,)))
        nn = None if nnghs is None else np.ascontiguousarray(np.broadcast_to(nnghs, (n,)), dtype=np.int32)
        check(lib.twxi_gwr_mth(self._h, C.byref(p), int(mth), ptr(nn), ptr(ptn), ptr(out), ptr(st), MEM_HOST))
        return out, st

    def xval_anom(self, stn_idx, nnghs):
        """twxi_xval_anom: leave-one-out GWR at the stations ``stn_idx`` (context indices) for every neighbour count of
        ``nnghs``.  Returns bias, mae, r2 [n, len(nnghs), 12] and status [n]."""
        stn_idx = np.ascontiguousarray(stn_idx, dtype=np.int32)
        nnghs = np.ascontiguousarray(nnghs, dtype=np.int32)
        n, nc = stn_idx.size, nnghs.size
        bias, mae, r2 = (np.empty((n, nc, 12)) for _ in range(3))
        st = np.empty(n, dtype=np.uint8)
        check(lib.twxi_xval_anom(self._h, n, ptr(stn_idx), nc, ptr(nnghs), ptr(bias), ptr(mae), ptr(r2), ptr(st), MEM_HOST))
        return bias, mae, r2, st

    def xval_overall(self, stn_idx, daily=False):
        """twxi_xval_overall: leave-one-out interpolation (kriged normal + GWR daily anomaly) at the stations ``stn_idx``
        (context indices), each left out with any co-located station, and its skill against the station's own
        observations.  Returns bias, mae, r2, norms, se [n, 12], status [n] and, with ``daily``, the dailies [n, ndays]
        (otherwise None: they stay on the device)."""
        stn_idx = np.ascontiguousarray(stn_idx, dtype=np.int32)
        n = stn_idx.size
        dly = np.empty((n, self.ndays)) if daily else None
        bias, mae, r2, norms, se = (np.empty((n, 12)) for _ in range(5))
        st = np.empty(n, dtype=np.uint8)
        check(lib.twxi_xval_overall(self._h, n, ptr(stn_idx), ptr(dly), ptr(norms), ptr(se), ptr(bias), ptr(mae), ptr(r2),
                                    ptr(st), MEM_HOST))
        return bias, mae, r2, norms, se, st, dly

    def interp_points(self, lat, lon, elev, tdi, lst, rm_idx=None, rm_zero=False, daily=True):
        p, keep = self._points(lat, lon, elev=elev, tdi=tdi, lst=lst, rm_idx=rm_idx, rm_zero=rm_zero)
        n = p.npts
        dly = np.empty((n, self.ndays)) if daily else None
        norms, se, var = np.empty((n, 12)), np.empty((n, 12)), np.empty((n, 12))
        st = np.empty(n, dtype=np.uint8)
        check(lib.twxi_interp_points(self._h, C.byref(p), ptr(dly), ptr(norms), ptr(se), ptr(var), ptr(st), MEM_HOST))
        return dly, norms, se, var, st


def interp_cells(ctx_tmin, ctx_tmax, lat, lon, elev, tdi, climdiv, lst_tmin, lst_tmax, rm_idx_tmin=None,
                 rm_idx_tmax=None, rm_zero=False, fix_invalid=True):
    """twxi_interp_cells.  ``rm_idx_tmin`` / ``rm_idx_tmax`` [ncells, n_rm] are CONTEXT-LOCAL station indices (-1 = none):
    the Tmin and Tmax station tables are different subsets of the DB, so a station has a different index in each."""
    lat = _f8(np.atleast_1d(lat)); n = lat.size
    lon, elev, tdi = _f8(np.atleast_1d(lon)), _f8(np.atleast_1d(elev)), _f8(np.atleast_1d(tdi))
    climdiv = None if climdiv is None else _f8(np.atleast_1d(climdiv))
    lst_tmin, lst_tmax = _f8(np.asarray(lst_tmin).reshape(n, 12)), _f8(np.asarray(lst_tmax).reshape(n, 12))
    n_rm = 0
    if rm_idx_tmin is not None or rm_idx_tmax is not None:
        ra = None if rm_idx_tmin is None else np.asarray(rm_idx_tmin, dtype=np.int32).reshape(n, -1)
        rb = None if rm_idx_tmax is None else np.asarray(rm_idx_tmax, dtype=np.int32).reshape(n, -1)
        n_rm = max(0 if ra is None else ra.shape[1], 0 if rb is None else rb.shape[1])

        def pad(r):
            o = -np.ones((n, n_rm), dtype=np.int32)
            if r is not None:
                o[:, :r.shape[1]] = r
            return o
        rm_idx_tmin, rm_idx_tmax = pad(ra), pad(rb)
    nd = ctx_tmin.ndays
    tmin, tmax = np.empty((n, nd)), np.empty((n, nd))
    o = [np.empty((n, 12)) for _ in range(4)]
    ninv = np.empty(n, dtype=np.int32)
    st = np.empty(n, dtype=np.uint8)
    check(lib.twxi_interp_cells(ctx_tmin.handle, ctx_tmax.handle, n, ptr(lat), ptr(lon), ptr(elev), ptr(tdi),
                                ptr(climdiv), ptr(lst_tmin), ptr(lst_tmax), ptr(rm_idx_tmin), ptr(rm_idx_tmax), n_rm,
                                int(bool(rm_zero)),
                                int(bool(fix_invalid)), ptr(tmin), ptr(tmax), ptr(o[0]), ptr(o[1]), ptr(o[2]),
                                ptr(o[3]), ptr(ninv), ptr(st), MEM_HOST))
    return tmin, tmax, o[0], o[1], o[2], o[3], ninv, st


def interp_chunk(ctx_tmin, ctx_tmax, wrk_chk, out=None, daily=True, wait=True):
    """twxi_interp_chunk on a work chunk ``f8[32, ny, nx]`` (numpy / pinned torch host tensor / CUDA tensor).
    ``out`` may carry preallocated result buffers (same memory space, dtypes and shapes are checked).  ``wait=False``
    submits the chunk with twxi_interp_chunk_async: its buffers belong to the library until ``interp_chunk_wait`` returns or
    until two further chunks have been submitted on the same context pair (the second submission blocks the host until this
    chunk's results are in the host buffers); the copies overlap the neighbouring chunks' kernels."""
    ny, nx = _check_wrk_chk(wrk_chk)
    if daily and ctx_tmin.ndays != ctx_tmax.ndays:
        raise ValueError("tmin and tmax contexts hold observation records of different length")
    nd = ctx_tmin.ndays
    dev = _lib.is_device(wrk_chk)
    want = dict(tmin=("int16", (nd, ny, nx)), tmax=("int16", (nd, ny, nx)), tmin_norm=("float32", (12, ny, nx)),
                tmax_norm=("float32", (12, ny, nx)), tmin_se=("float32", (12, ny, nx)), tmax_se=("float32", (12, ny, nx)),
                ninvalid=("int32", (ny, nx)), status=("uint8", (ny, nx)))
    if not daily:                                             # normals only: tmin / tmax may be absent
        want = {k: v for k, v in want.items() if k not in ("tmin", "tmax") or (out or {}).get(k) is not None}
    bufs, _ = _result_buffers(want, out, wrk_chk.device if dev else None, wrk_dev=dev)
    out = dict(tmin=None, tmax=None, **bufs) if out is None and not daily else bufs
    fn = lib.twxi_interp_chunk if wait else lib.twxi_interp_chunk_async
    check(fn(ctx_tmin.handle, ctx_tmax.handle, ptr(wrk_chk), int(ny), int(nx),
             ptr(out["tmin"]), ptr(out["tmax"]), ptr(out["tmin_norm"]), ptr(out["tmax_norm"]),
             ptr(out["tmin_se"]), ptr(out["tmax_se"]), ptr(out["ninvalid"]), ptr(out["status"]),
             MEM_DEVICE if dev else MEM_HOST))
    return out


def interp_chunk_wait(ctx_tmin, host_sync=True):
    """Completion of the chunks submitted with ``interp_chunk(..., wait=False)`` (twxi_interp_chunk_wait)."""
    check(lib.twxi_interp_chunk_wait(ctx_tmin.handle, 1 if host_sync else 0))


def _check_wrk_chk(wrk_chk):
    if len(wrk_chk.shape) != 3 or wrk_chk.shape[0] != 32:
        raise ValueError("wrk_chk must be [32, ny, nx] (planes of tiling.py:205-213 / step25:273-279), got %r"
                         % (tuple(wrk_chk.shape),))
    if _dtype_name(wrk_chk) != "float64":
        raise ValueError("wrk_chk must be float64, got %s" % _dtype_name(wrk_chk))
    return int(wrk_chk.shape[1]), int(wrk_chk.shape[2])


def _result_buffers(want, out, device, wrk_dev=None):
    """Result buffers {name: (dtype, shape)}: allocated when ``out`` is None (numpy on the host, or torch tensors on the CUDA
    ``device``), otherwise checked (dtype, shape, one memory space: that of wrk_chk when ``wrk_dev`` gives it).  Returns
    (buffers, on_device)."""
    if out is None:
        if device is None:
            return {k: np.empty(shp, dtype=dt) for k, (dt, shp) in want.items()}, False
        import torch
        return {k: torch.empty(shp, dtype=getattr(torch, dt), device=device) for k, (dt, shp) in want.items()}, True
    dev = wrk_dev
    for k, (dt, shp) in want.items():
        b = out.get(k)
        if b is None:
            raise ValueError("out[%r] is missing" % k)
        if _dtype_name(b) != dt or tuple(b.shape) != shp:
            raise ValueError("out[%r] must be %s %r, got %s %r" % (k, dt, shp, _dtype_name(b), tuple(b.shape)))
        if dev is None:
            dev = _lib.is_device(b)
        elif _lib.is_device(b) != dev:
            raise ValueError("out[%r] must live in the same memory space as %s"
                             % (k, "the other result buffers" if wrk_dev is None else "wrk_chk"))
    return out, dev


def _check_unpinned(bufs):
    """Host torch tensors handed to an asynchronous call must be pinned: the copy stream reads or writes them after the call
    returns."""
    for k, b in bufs.items():
        if b is not None and hasattr(b, "is_pinned") and not b.is_cuda and not b.is_pinned():
            raise ValueError("%s is a torch host tensor that is not pinned: wait=False needs pinned host buffers "
                             "(tensor.pin_memory())" % k)


def _async_results(want, out, device, wait):
    """_result_buffers for the tile calls.  wait=False with host results needs the caller's ``out``: the library owns those
    buffers until two further submissions, so none is allocated behind the caller's back."""
    if not wait:
        if out is None and device is None:
            raise ValueError("wait=False with host buffers needs `out`: the buffers belong to the library until two "
                             "further submissions (or interp_chunk_wait), so the caller has to own them")
        if out is not None:
            _check_unpinned(out)
    return _result_buffers(want, out, device)


def tile_begin(ctx_tmin, ctx_tmax, wrk_chk, wait=True):
    """twxi_tile_begin: everything of interp_chunk that does not depend on the day (kNN, neighbour counts, kriging, GWR hat
    rows) for the work chunk ``wrk_chk`` f8[32, ny, nx]; opens a tile on the context pair.  Returns (ny, nx).
    ``wait=False`` submits it with twxi_tile_begin_async: a host ``wrk_chk`` (pinned, for the overlap) belongs to the
    library until ``interp_chunk_wait`` returns or two further submissions have been made on the pair."""
    ny, nx = _check_wrk_chk(wrk_chk)
    if ctx_tmin.ndays != ctx_tmax.ndays:
        raise ValueError("tmin and tmax contexts hold observation records of different length")
    if not wait:
        _check_unpinned(dict(wrk_chk=wrk_chk))
    fn = lib.twxi_tile_begin if wait else lib.twxi_tile_begin_async
    check(fn(ctx_tmin.handle, ctx_tmax.handle, ptr(wrk_chk), ny, nx, MEM_DEVICE if _lib.is_device(wrk_chk) else MEM_HOST))
    return ny, nx


def tile_days(ctx_tmin, ctx_tmax, ndays, shape, out=None, device=None, wait=True):
    """twxi_tile_days: the next ``ndays`` days of the open tile of ``shape`` = (ny, nx) -> {tmin, tmax} int16
    [ndays, ny, nx], byte-identical to the same days of interp_chunk.  ``out`` may carry the two buffers; otherwise they are
    allocated on the host, or on the CUDA ``device`` (a torch device) when given.  ``wait=False`` submits the window with
    twxi_tile_days_async; host buffers must then come in ``out`` (pinned torch tensors, or numpy arrays without overlap)
    and belong to the library until ``interp_chunk_wait`` returns or two further submissions have been made on the pair."""
    ny, nx = shape
    want = dict(tmin=("int16", (int(ndays), ny, nx)), tmax=("int16", (int(ndays), ny, nx)))
    out, dev = _async_results(want, out, device, wait)
    fn = lib.twxi_tile_days if wait else lib.twxi_tile_days_async
    check(fn(ctx_tmin.handle, ctx_tmax.handle, int(ndays), ptr(out["tmin"]), ptr(out["tmax"]),
             MEM_DEVICE if dev else MEM_HOST))
    return out


class MonthGroups(object):
    """The month runs of the record's days table (db.month_runs) and `day0`, the first day of the next window of the open
    tile: tile_days_mth reads the runs a window completes from it and advances it.  Make one after each tile_begin."""

    def __init__(self, days):
        self.start, self.ndays, self.year, self.month = db.month_runs(days)
        self.day0 = 0

    def completed(self, n):
        """Indices [g0, g1) of the runs whose last day falls in the days day0 .. day0 + n - 1."""
        ends = self.start + self.ndays
        return int(np.searchsorted(ends, self.day0, side="right")), int(np.searchsorted(ends, self.day0 + n, side="right"))


def tile_days_mth(ctx_tmin, ctx_tmax, ndays, shape, groups, out=None, device=None, wait=True):
    """twxi_tile_days_mth: tile_days plus the monthly means of every month run that ends in the window ->
    {tmin, tmax} int16 [ndays, ny, nx], {tmin_mth, tmax_mth} float32 [nmth, ny, nx] and mth_groups, the (year, month,
    ndays) of each month, chronological.  ``groups`` is the MonthGroups of the tile (advanced by ndays); the month count
    is exact, so ``out``'s month buffers must be [nmth, ny, nx].  ``wait=False``: twxi_tile_days_mth_async, with the
    buffer rules of tile_days; the month count and mth_groups are known at return."""
    ny, nx = shape
    g0, g1 = groups.completed(int(ndays))
    nm = g1 - g0
    want = dict(tmin=("int16", (int(ndays), ny, nx)), tmax=("int16", (int(ndays), ny, nx)),
                tmin_mth=("float32", (nm, ny, nx)), tmax_mth=("float32", (nm, ny, nx)))
    out, dev = _async_results(want, out, device, wait)
    n = C.c_int32(-1)
    fn = lib.twxi_tile_days_mth if wait else lib.twxi_tile_days_mth_async
    check(fn(ctx_tmin.handle, ctx_tmax.handle, int(ndays), ptr(out["tmin"]), ptr(out["tmax"]), nm,
             ptr(out["tmin_mth"]) if nm else None, ptr(out["tmax_mth"]) if nm else None, C.byref(n),
             MEM_DEVICE if dev else MEM_HOST))
    if n.value != nm:
        raise RuntimeError("twxi_tile_days_mth completed %d months, the days table %d" % (n.value, nm))
    groups.day0 += int(ndays)
    out["mth_groups"] = [(int(groups.year[g]), int(groups.month[g]), int(groups.ndays[g])) for g in range(g0, g1)]
    return out


def tile_end(ctx_tmin, ctx_tmax, shape, out=None, device=None, wait=True):
    """twxi_tile_end after the last day: {tmin_norm, tmax_norm, tmin_se, tmax_se, ninvalid, status} of interp_chunk
    (normals recomputed from the fixed 1981-2010 dailies when a day was fixed); closes the tile.  ``wait=False``:
    twxi_tile_end_async, with the buffer rules of tile_days; the tile is closed at return, so the next tile_begin may
    follow at once."""
    ny, nx = shape
    want = dict(tmin_norm=("float32", (12, ny, nx)), tmax_norm=("float32", (12, ny, nx)),
                tmin_se=("float32", (12, ny, nx)), tmax_se=("float32", (12, ny, nx)),
                ninvalid=("int32", (ny, nx)), status=("uint8", (ny, nx)))
    out, dev = _async_results(want, out, device, wait)
    fn = lib.twxi_tile_end if wait else lib.twxi_tile_end_async
    check(fn(ctx_tmin.handle, ctx_tmax.handle, ptr(out["tmin_norm"]), ptr(out["tmax_norm"]),
             ptr(out["tmin_se"]), ptr(out["tmax_se"]), ptr(out["ninvalid"]), ptr(out["status"]),
             MEM_DEVICE if dev else MEM_HOST))
    return out

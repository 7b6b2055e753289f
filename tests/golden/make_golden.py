"""Generate the committed golden vectors from the REFERENCE'S OWN CODE (run in the build container).

    python tests/golden/make_golden.py

Uses ``oracle.ref_loader`` to execute, unmodified, from ``/root/reference``:
``grt_circle_dist`` (twx/utils/util_geo.py:24-40), ``StationSelect`` (twx/interp/station_select.py),
``_gwr_series`` (twx/interp/interp_tair.py:1099-1146) and ``tmin_tmax_fixer`` (:143-197) on seeded
synthetic inputs, and stores inputs + outputs in ``tests/golden/*.npz``.  The reference tree is not
available on the GPU box, so tests read only the ``.npz`` files.  The kriging half of the path runs in
R/gstat and cannot be executed here: no golden vectors exist for it (see oracle/__init__.py).
"""
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import ref_loader          # noqa: E402
from topowx_b200 import synth, db      # noqa: E402

warnings.simplefilter("ignore", DeprecationWarning)


def small_db(which=0, n=600):
    f = synth.Fields()
    days = synth.make_days(1995, 1)
    return synth.make_station_db(which, n, synth.tile_bbox(buf=1.5), f, days), f


def main():
    ref = ref_loader.load()
    rng = np.random.default_rng(12345)

    # ---- grt_circle_dist ---------------------------------------------------------------------
    lon1, lat1 = rng.uniform(-125, -67, 2000), rng.uniform(24, 50, 2000)
    lon2, lat2 = lon1 + rng.normal(0, 2, 2000), lat1 + rng.normal(0, 2, 2000)
    lon2[:10], lat2[:10] = lon1[:10], lat1[:10]                       # zero distances
    np.savez(os.path.join(HERE, "grt_circle_dist.npz"), lon1=lon1, lat1=lat1, lon2=lon2, lat2=lat2,
             dist=ref.grt_circle_dist(lon1, lat1, lon2, lat2))

    # ---- StationSelect ------------------------------------------------------------------------
    stn_da, f = small_db()
    good = np.isnan(stn_da.stns[db.BAD])
    gidx = np.nonzero(good)[0]
    cases = []
    ss = ref.StationSelect(stn_da, good)
    ss_rm0 = ref.StationSelect(stn_da, good, rm_zero_dist_stns=True)
    pts_lat = rng.uniform(39.7, 41.6, 24)
    pts_lon = rng.uniform(-99.9, -98.0, 24)
    out = dict(stn_lon=stn_da.stns[db.LON], stn_lat=stn_da.stns[db.LAT], good=good)
    idx_all, d_all, w_all, meta = [], [], [], []
    for i, (la, lo) in enumerate(zip(pts_lat, pts_lon)):
        for nn in (35, 100, 147):
            ss.set_ngh_stns(la, lo, nn, load_obs=False)
            ids = ss.ngh_stns[db.STN_ID]
            idx_all.append(np.array([stn_da.stn_idxs[s] for s in ids]))
            d_all.append(ss.ngh_dists.copy()); w_all.append(ss.ngh_wgt.copy())
            meta.append((la, lo, nn, -1, 0))
    # leave-one-out at station locations (optimize.py:569,602-603): stns_rm = own id, zero-dist removal
    for s in gidx[rng.choice(gidx.size, 12, replace=False)]:
        st = stn_da.stns[s]
        for nn in (35, 100):
            ss_rm0.set_ngh_stns(st[db.LAT], st[db.LON], nn, load_obs=False, stns_rm=st[db.STN_ID])
            ids = ss_rm0.ngh_stns[db.STN_ID]
            idx_all.append(np.array([stn_da.stn_idxs[x] for x in ids]))
            d_all.append(ss_rm0.ngh_dists.copy()); w_all.append(ss_rm0.ngh_wgt.copy())
            meta.append((st[db.LAT], st[db.LON], nn, s, 1))
    # obs loading order (station_select.py:184-185 -> DB order); the station table's obs are stored for January-August
    # only (the case reads March), which keeps the file under 1 MB
    ss.set_ngh_stns(pts_lat[0], pts_lon[0], 40, load_obs=True, obs_mth=3)
    month = np.asarray(stn_da.days[db.MONTH])
    out.update(obs_case_idx=np.array([stn_da.stn_idxs[s] for s in ss.ngh_stns[db.STN_ID]]),
               obs_case=ss.ngh_obs, obs_all=stn_da.var[month <= 8], month=month[month <= 8])
    K = max(len(a) for a in idx_all)
    pad = lambda a, fill: np.array([np.concatenate([x, np.full(K - len(x), fill)]) for x in a])
    out.update(meta=np.array(meta, dtype=np.float64), idx=pad(idx_all, -1).astype(np.int64),
               dists=pad(d_all, np.nan), wgt=pad(w_all, np.nan))
    np.savez(os.path.join(HERE, "station_select.npz"), **out)

    # ---- _gwr_series --------------------------------------------------------------------------
    g = {}
    for c in range(6):
        k = int(rng.choice([35, 57, 101, 147]))
        X = np.column_stack([rng.uniform(-101, -97, k), rng.uniform(38, 43, k), rng.uniform(200, 2500, k),
                             rng.uniform(0, 1, k), rng.normal(10, 6, k)])
        x = np.array([-99.0, 40.5, 900.0, 0.4, 11.0]) + rng.normal(0, 0.1, 5)
        y = (rng.normal(0, 4, (31, k))).astype(np.float32).astype(np.float64)
        d = np.sort(rng.uniform(1, 150, k + 1))
        w = np.square(1.0 - np.square(d[:k] / d[k]))
        g["X%d" % c], g["x%d" % c], g["y%d" % c], g["w%d" % c] = X, x, y, w
        g["p%d" % c] = ref._gwr_series(X, x, y, w)
    np.savez(os.path.join(HERE, "gwr_series.npz"), **g)

    # ---- tmin_tmax_fixer ----------------------------------------------------------------------
    fx = {}
    for c in range(5):
        n = 365
        tmin = rng.normal(5, 6, n)
        tmax = tmin + rng.normal(2.0, 2.5, n)
        if c == 0:
            tmax = tmin + np.abs(rng.normal(3, 1, n)) + 0.1          # nothing to fix
        if c == 4:
            tmax[:5] = tmin[:5] - 1.0                                 # fixes at the array start
        a, b, ninv = ref.tmin_tmax_fixer(tmin, tmax)
        fx["tmin%d" % c], fx["tmax%d" % c], fx["otmin%d" % c], fx["otmax%d" % c], fx["ninv%d" % c] = tmin, tmax, a, b, ninv
    np.savez(os.path.join(HERE, "tmin_tmax_fixer.npz"), **fx)
    print("golden vectors written to", HERE)


if __name__ == "__main__":
    main()

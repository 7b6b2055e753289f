"""Pin the numpy oracle against golden vectors produced by the reference's own code
(tests/golden/make_golden.py executes util_geo.py / station_select.py / _gwr_series / tmin_tmax_fixer
verbatim from the original TopoWx sources).  CPU only."""
import os

import numpy as np

from oracle import twx_oracle as o


def _mini_db(g):
    n = g["stn_lon"].size
    stns = np.zeros(n, dtype=[(o.STN_ID, "U16"), (o.LON, "f8"), (o.LAT, "f8"), (o.BAD, "f8")])
    stns[o.STN_ID] = ["SYN%06d" % i for i in range(n)]
    stns[o.LON], stns[o.LAT] = g["stn_lon"], g["stn_lat"]
    stns[o.BAD] = np.where(g["good"], np.nan, 1.0)
    days = np.zeros(g["month"].size, dtype=[(o.YEAR, "i4"), (o.MONTH, "i4")])
    days[o.MONTH] = g["month"]
    days[o.YEAR] = 1995
    return o.StationDb(stns, g["obs_all"], days)


def test_grt_circle_dist_bit_exact(golden_dir):
    g = np.load(os.path.join(golden_dir, "grt_circle_dist.npz"))
    d = o.grt_circle_dist(g["lon1"], g["lat1"], g["lon2"], g["lat2"])
    assert np.array_equal(d, g["dist"])
    assert np.all(d[:10] == 0)


def test_station_select_matches_reference(golden_dir):
    g = np.load(os.path.join(golden_dir, "station_select.npz"))
    sd = _mini_db(g)
    good = g["good"]
    ss = o.StationSelect(sd, good)
    ss0 = o.StationSelect(sd, good, rm_zero_dist_stns=True)
    for meta, idx, d, w in zip(g["meta"], g["idx"], g["dists"], g["wgt"]):
        lat, lon, nn, rm, rm0 = meta[0], meta[1], int(meta[2]), int(meta[3]), int(meta[4])
        sel = ss0 if rm0 else ss
        sel.set_ngh_stns(lat, lon, nn, load_obs=False, stns_rm=None if rm < 0 else sd.stn_ids[rm])
        gi = sel.stn_gidx[sel.ngh_idx]
        assert np.array_equal(gi, idx[:nn])                 # neighbour indices bit-exact, id order
        assert np.array_equal(sel.ngh_dists, d[:nn])        # same numpy arithmetic -> bit-exact
        assert np.array_equal(sel.ngh_wgt, w[:nn])
        if rm >= 0:
            assert rm not in gi
    # no exact distance ties in the fixture: the stable tie-break cannot differ from the reference's sort
    ss._set_pt(g["meta"][0][0], g["meta"][0][1])
    assert np.unique(ss.pt_sort_stn_dists).size == ss.pt_sort_stn_dists.size


def test_station_select_obs_order(golden_dir):
    g = np.load(os.path.join(golden_dir, "station_select.npz"))
    sd = _mini_db(g)
    ss = o.StationSelect(sd, g["good"])
    ss.set_ngh_stns(g["meta"][0][0], g["meta"][0][1], 40, load_obs=True, obs_mth=3)
    assert np.array_equal(ss.stn_gidx[ss.ngh_idx], g["obs_case_idx"])
    assert np.array_equal(ss.ngh_obs, g["obs_case"])


def test_gwr_series_matches_reference(golden_dir):
    g = np.load(os.path.join(golden_dir, "gwr_series.npz"))
    for c in range(6):
        p, z = o.gwr_series(g["X%d" % c], g["x%d" % c], g["y%d" % c], g["w%d" % c])
        # same algebra (inv of X'WX); diag(w) product replaced by a broadcast -> rounding-level only
        np.testing.assert_allclose(p, g["p%d" % c], rtol=0, atol=2e-9)
        assert abs(z.sum() - 1.0) < 1e-8


def test_fixer_matches_reference(golden_dir):
    g = np.load(os.path.join(golden_dir, "tmin_tmax_fixer.npz"))
    for c in range(5):
        a, b, n = o.tmin_tmax_fixer(g["tmin%d" % c], g["tmax%d" % c])
        assert n == int(g["ninv%d" % c])
        assert np.array_equal(a, g["otmin%d" % c]) and np.array_equal(b, g["otmax%d" % c])
    assert int(g["ninv0"]) == 0 and int(g["ninv4"]) >= 5

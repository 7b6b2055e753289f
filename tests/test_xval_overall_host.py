"""Host side of the step-24 skill figures (twxi_xval_overall), CPU only: the statistics the kernel computes, restated in
numpy from the oracle's leave-one-out interpolation, and the arguments of scripts/step24_xval_interp.py."""
import importlib.util
import os

import numpy as np
import pytest
from scipy import stats

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _kernel_stats(x, y, ns):
    """xval_stats_kernel in numpy: anomalies from the station's normal ns, lane partial sums in day order (lane = day mod
    32), the shuffle tree of warp_sum, then the centred-sum statistics."""
    x, y = x - ns, y - ns
    D = x.size

    def lane_sums(v):
        p = np.zeros(32)
        for d in range(D):
            p[d % 32] += v[d]
        for off in (16, 8, 4, 2, 1):
            p = p + p[np.arange(32) ^ off]
        return p[0]
    sd, sad, sx, sy = lane_sums(x - y), lane_sums(np.abs(x - y)), lane_sums(x), lane_sums(y)
    sxx, syy, sxy = lane_sums(x * x), lane_sums(y * y), lane_sums(x * y)
    n = float(D)
    cxy, cxx, cyy = sxy - sx * sy / n, sxx - sx * sx / n, syy - sy * sy / n
    r = cxy / np.sqrt(cxx * cyy)
    return sd / n, sad / n, r * r


def test_kernel_statistics_of_oracle_interpolation():
    """The kernel's statistics of the oracle's leave-one-out dailies (oracle.XvalTairOverall.run_interp) against the
    station's observations (load_obs) equal the definitions of XvalTairAnom.run_xval: mean, mean absolute value and
    scipy.stats.linregress r^2."""
    from oracle import twx_oracle as o
    from topowx_b200 import synth, db
    da = synth.make_station_db(0, 150, synth.tile_bbox(buf=1.0), synth.Fields(), synth.make_days(1995, 1))
    oda = o.StationDb(da.stns, da.var, da.days)
    oxv = o.XvalTairOverall(oda)
    good = np.nonzero(np.isnan(da.stns[db.BAD]) & np.isfinite(da.stns[db.MASK]))[0]
    sid = da.stns[db.STN_ID][good[11]]
    dly, _, _ = oxv.run_interp(sid)
    obs = oda.load_obs(np.array([sid]))[:, 0].astype(np.float64)
    stn = oda.stns[oda.stn_idxs[sid]]
    for mth in (1, 6, 11):
        i = oda.mth_idx[mth]
        x, y = dly[i], obs[i]
        bias, mae, r2 = _kernel_stats(x, y, stn[db.get_norm_varname(mth)])
        assert abs(bias - np.mean(x - y)) < 1e-12
        assert abs(mae - np.mean(np.abs(x - y))) < 1e-12
        assert abs(r2 - stats.linregress(x, y)[2] ** 2) < 1e-12
        assert abs(r2 - np.corrcoef(x, y)[0, 1] ** 2) < 1e-12


def test_anomaly_sums_hold_r2_over_a_long_record():
    """Over the ~2 100 days a month has in a 68-year record the raw sums cancel ~20 C means; the anomalies from the
    station's normal keep r^2 to 1e-9 of linregress."""
    rng = np.random.default_rng(5)
    n = 2108
    y = (21.3 + rng.normal(0, 3, n)).astype(np.float32).astype(np.float64)
    x = y + rng.normal(0, 1.2, n)
    ref = stats.linregress(x, y)[2] ** 2
    assert abs(_kernel_stats(x, y, 21.27)[2] - ref) < 1e-9


def _step24():
    path = os.path.join(ROOT, "scripts", "step24_xval_interp.py")
    spec = importlib.util.spec_from_file_location("step24_xval_interp", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_step24_arguments():
    s = _step24()
    a = s.parse_args(["tmin"])
    assert (a.year0, a.years, a.stats, a.daily, a.batch) == (1995, 1, False, False, 4096)
    a = s.parse_args(["tmax", "--year0", "1948", "--years", "68", "--stats", "--daily", "--out", "x.npz"])
    assert (a.elem, a.year0, a.years, a.stats, a.daily, a.out) == ("tmax", 1948, 68, True, True, "x.npz")
    for bad in (["tmin", "--daily"], ["tmin", "--years", "0"], ["tavg"]):
        with pytest.raises(SystemExit):
            s.parse_args(bad)

"""Step 24 over a multi-decade record: the skill figures computed on the device against the dailies shipped to the host.

    python tools/xval_record.py [--year0 1948] [--years 68] [--nstns 10000] [--batch 4096] [--passes 2]

One variable (tmin) of the 10 000-station C5 table (bench.py) over a seeded synthetic record (default 1948-2015, 24 837
days); the cross-validation stations are the in-domain, non-bad ones (step24:133-135), in batches of --batch.  Two paths,
alternated over --passes passes after one warm-up pass each, every batch timed with a host clock around calls that end in
a device synchronise:
    device  twxi_xval_overall with daily = NULL: bias / MAE / r^2 [n, 12] are computed on the device and only they, the
            normals and the status leave it;
    host    twxi_interp_points (rm_idx = the station, rm_zero_dist = 1) with the dailies copied to the host, then the same
            statistics in numpy against the observation table.
Prints one JSON line with the device name and power limit (read-only nvidia-smi query), the per-pass times of both paths,
and the largest difference between the two paths' statistics and normals.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np                                                              # noqa: E402

import bench                                                                    # noqa: E402
from record_tile import gpu_name_power                                          # noqa: E402
from topowx_b200 import db, synth                                               # noqa: E402
from topowx_b200.context import TwxiContext                                     # noqa: E402


def numpy_stats(dly, obs, mth_idx):
    """bias, MAE, r^2 [n, 12] of dly [n, ndays] against obs [n, ndays] over every day of each month."""
    n = dly.shape[0]
    out = np.full((3, n, 12), np.nan)
    for m in range(1, 13):
        i = mth_idx[m]
        if i.size == 0:
            continue
        x, y = dly[:, i], obs[:, i]
        out[0, :, m - 1] = np.mean(x - y, axis=1)
        out[1, :, m - 1] = np.mean(np.abs(x - y), axis=1)
        xm, ym = x - x.mean(axis=1, keepdims=True), y - y.mean(axis=1, keepdims=True)
        with np.errstate(all="ignore"):
            out[2, :, m - 1] = ((xm * ym).sum(1) / np.sqrt((xm * xm).sum(1) * (ym * ym).sum(1))) ** 2
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--year0", type=int, default=1948)
    ap.add_argument("--years", type=int, default=68)
    ap.add_argument("--nstns", type=int, default=bench.NSTNS_C5)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--passes", type=int, default=2)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("xval_record.py measures on a CUDA device; none is available")
    torch.cuda.set_device(args.device)
    name, power = gpu_name_power(args.device)

    days = synth.make_days(args.year0, args.years)
    da = synth.make_station_db(0, args.nstns, synth.conus_bbox(1.0), synth.Fields(), days, seed=synth.SEED_STNS)
    good = np.isnan(da.stns[db.BAD])
    ctx = TwxiContext(da, good, device=args.device)
    sel = np.nonzero(good & np.isfinite(da.stns[db.MASK]))[0]
    loc = ctx.local_of_db[sel].astype(np.int32)
    s = da.stns[sel]
    lst = np.stack([s[db.get_lst_varname(m)] for m in range(1, 13)], axis=1)
    batches = [slice(i, min(i + args.batch, sel.size)) for i in range(0, sel.size, args.batch)]

    def run_device():
        return [ctx.xval_overall(loc[b]) for b in batches]

    def run_host():
        res = []
        for b in batches:
            dly, norms, se, var, st = ctx.interp_points(s[db.LAT][b], s[db.LON][b], s[db.ELEV][b], s[db.TDI][b], lst[b],
                                                        rm_idx=loc[b, None], rm_zero=True)
            obs = np.asarray(da.var[:, sel[b]], dtype=np.float64).T
            bias, mae, r2 = numpy_stats(dly, obs, da.mth_idx)
            bad = st != 0
            for a in (bias, mae, r2):
                a[bad] = np.nan
            res.append((bias, mae, r2, norms, se, st))
        return res

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0, r

    _, dev_res = timed(run_device)                         # warm-up passes
    _, host_res = timed(run_host)
    t_dev, t_host = [], []
    for _ in range(args.passes):
        t_dev.append(timed(run_device)[0])
        t_host.append(timed(run_host)[0])

    diff = {}
    for k, name_ in enumerate(("bias", "mae", "r2", "norms")):
        a = np.concatenate([r[k] for r in dev_res])
        b = np.concatenate([r[k] for r in host_res])
        ok = np.concatenate([r[5] for r in dev_res]) == 0
        diff[name_] = float(np.nanmax(np.abs(a[ok] - b[ok]))) if ok.any() else None
    st = np.concatenate([r[5] for r in dev_res])
    st_host = np.concatenate([r[5] for r in host_res])
    mae = np.concatenate([r[1] for r in dev_res])[st == 0]
    res = dict(tool="xval_record", device=name, power_limit=power, stations=int(sel.size), table=int(ctx.n),
               days=int(days.size), years="%d-%d" % (args.year0, args.year0 + args.years - 1), batch=args.batch,
               device_path_ms=[round(t * 1e3, 2) for t in t_dev], host_path_ms=[round(t * 1e3, 1) for t in t_host],
               daily_bytes_not_copied=int(sel.size) * int(days.size) * 8,
               failed=int((st != 0).sum()), status_equal=bool(np.array_equal(st, st_host)),
               max_abs_diff=diff, median_mae_by_month=[round(float(v), 4) for v in np.median(mae, axis=0)])
    print(json.dumps(res))


if __name__ == "__main__":
    main()

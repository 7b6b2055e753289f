#!/usr/bin/env python
'''
Leave-one-out cross validation driver: the Python-3 / GPU counterpart of scripts/step24_mpi_xval_interp.py.

    python scripts/step24_xval_interp.py tmin|tmax [--nstns 10000] [--max-stations 2000] [--year0 1995 --years 1]
                                         [--stats [--daily]] [--out xval.npz]
    torchrun --nproc-per-node N scripts/step24_xval_interp.py tmax ...

The reference sends one station id per MPI message to idle workers (step24:130-156).  Here the in-domain,
non-bad stations (step24:133-135) are split contiguously over the ranks and each rank interpolates its share
with XvalTairOverall.run_interp_batch (one twxi_interp_points call per batch of stations), or with --stats
XvalTairOverall.run_xval_batch (one twxi_xval_overall call per batch): bias, MAE and r^2 per station and month are
computed on the device, and the daily series leave it only with --daily.  The synthetic record covers the years
year0 .. year0 + years - 1.  Each rank prints one summary line (with --stats: the median MAE of each month).
'''
import argparse
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from topowx_b200 import synth, db                       # noqa: E402
from topowx_b200.interp import XvalTairOverall          # noqa: E402


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("elem", choices=["tmin", "tmax"])
    ap.add_argument("--nstns", type=int, default=10000)
    ap.add_argument("--max-stations", type=int, default=0, help="limit the number of xval stations (0 = all)")
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--year0", type=int, default=1995, help="first year of the synthetic record")
    ap.add_argument("--years", type=int, default=1, help="length of the synthetic record in years")
    ap.add_argument("--stats", action="store_true", help="bias / MAE / r^2 per station and month, computed on the GPU")
    ap.add_argument("--daily", action="store_true", help="with --stats: also return and write the daily series")
    ap.add_argument("--out", default="")
    args = ap.parse_args(argv)
    if args.years < 1:
        ap.error("--years must be >= 1")
    if args.daily and not args.stats:
        ap.error("--daily goes with --stats (without --stats the daily series are always written)")
    return args


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    which = 0 if args.elem == "tmin" else 1
    days = synth.make_days(args.year0, args.years)
    stn_da = synth.make_station_db(which, args.nstns, synth.conus_bbox(), synth.Fields(), days)
    xval = XvalTairOverall(stn_da, args.elem, device=local_rank)
    stn_mask = np.logical_and(np.isfinite(stn_da.stns[db.MASK]), np.isnan(stn_da.stns[db.BAD]))
    ids = stn_da.stn_ids[stn_mask]
    if args.max_stations:
        ids = ids[:args.max_stations]
    mine = np.array_split(ids, world)[rank]
    t0 = time.time()
    res = dict(norms=[], se=[], status=[], daily=[], bias=[], mae=[], r2=[])
    for i in range(0, mine.size, args.batch):
        batch = mine[i:i + args.batch]
        if args.stats:
            r = xval.run_xval_batch(batch, daily=args.daily)
            for k, v in zip(("bias", "mae", "r2", "norms", "se", "status", "daily"), r):
                res[k].append(v)
        else:
            dly, nrm, se, st = xval.run_interp_batch(batch)
            for k, v in zip(("daily", "norms", "status"), (dly, nrm, st)):
                res[k].append(v)
    dt = time.time() - t0
    res = {k: np.concatenate(v) for k, v in res.items() if v}
    status = res.get("status", np.zeros(0, np.uint8))
    line = ("rank %d/%d: %d stations x 12 months x %d days in %.2f s; %d failed"
            % (rank, world, mine.size, days.size, dt, int((status != 0).sum())))
    if args.stats:
        ok = res["mae"][status == 0] if mine.size else np.full((0, 12), np.nan)
        med = np.nanmedian(ok, axis=0) if ok.shape[0] else np.full(12, np.nan)
        line += "; median MAE by month (C): " + " ".join("%.3f" % v for v in med)
    print(line)
    if args.out:
        np.savez_compressed("%s.rank%d" % (args.out, rank), stn_ids=mine, **res)


if __name__ == "__main__":
    main()

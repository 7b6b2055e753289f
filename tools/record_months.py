"""Cost of the monthly means (twxi_tile_days_mth) on one full-land C5 tile over a multi-decade record, in year windows.

    python tools/record_months.py [--year0 1948] [--years 68] [--nstns 10000] [--reps 3]

The record is synthetic and seeded, the tile and station table are tools/record_tile.py's.  Prints one JSON line:
  * device name and power limit (read-only nvidia-smi query);
  * the whole stream (twxi_tile_begin, 68 year windows, twxi_tile_end) with device buffers, with twxi_tile_days and with
    twxi_tile_days_mth: CUDA events around each pass, the two alternated `--reps` times after a warm-up pass of each;
  * tile_month_kernel's device time per window and in total, from torch.profiler (CUDA activities) in a pass of its own,
    with the window's tile_apply_kernel and tile_fix_kernel times beside it;
  * the host time numpy takes for the same grids from the int16 record already in host memory (exact int sums per month
    run, the contract's expression), which is the reduction a user of the daily files runs today, without reading them;
  * whether the GPU grids equal numpy's bit for bit, and whether the dailies of both passes are byte-identical.
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
from topowx_b200.context import (TwxiContext, tile_begin, tile_days, tile_days_mth, tile_end,   # noqa: E402
                                 MonthGroups)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--year0", type=int, default=1948)
    ap.add_argument("--years", type=int, default=68)
    ap.add_argument("--nstns", type=int, default=bench.NSTNS_C5)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("record_months.py measures on a CUDA device; none is available")
    torch.cuda.set_device(args.device)
    dev = torch.device("cuda", args.device)
    name, power = gpu_name_power(args.device)

    f, _, tiles, _ = bench.c5_tile_list(64)
    _, r0, c0, land = tiles[0]
    days = synth.make_days(args.year0, args.years)
    nd = int(days.size)
    yrs = np.unique(days[db.YEAR], return_counts=True)[1].tolist()
    start, ndays, _, _ = db.month_runs(days)
    da = [synth.make_station_db(w, args.nstns, synth.conus_bbox(1.0), f, days, seed=synth.SEED_STNS) for w in (0, 1)]
    ctx = [TwxiContext(d, np.isnan(d.stns[db.BAD]), device=args.device) for d in da]
    del da
    T = bench.TILE
    wrk = torch.from_numpy(synth.make_wrk_chk_grid(f, r0, c0, T, T)).to(dev)
    shape = (T, T)
    stream = torch.cuda.current_stream(dev)
    mk = lambda n, dt: torch.empty((n, T, T), dtype=dt, device=dev)
    dly = {m: dict(tmin=mk(nd, torch.int16), tmax=mk(nd, torch.int16)) for m in (False, True)}
    mth = dict(tmin_mth=mk(start.size, torch.float32), tmax_mth=mk(start.size, torch.float32))
    fin = {m: dict(tmin_norm=mk(12, torch.float32), tmax_norm=mk(12, torch.float32), tmin_se=mk(12, torch.float32),
                   tmax_se=mk(12, torch.float32), ninvalid=torch.empty(shape, dtype=torch.int32, device=dev),
                   status=torch.empty(shape, dtype=torch.uint8, device=dev)) for m in (False, True)}

    def one_pass(months):
        """begin, the year windows, end; device time from CUDA events on the contexts' stream."""
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        tile_begin(ctx[0], ctx[1], wrk)
        g = MonthGroups(days) if months else None
        d0 = m0 = 0
        for n in yrs:
            out = dict(tmin=dly[months]["tmin"][d0:d0 + n], tmax=dly[months]["tmax"][d0:d0 + n])
            if months:
                g0, g1 = g.completed(n)
                out.update(tmin_mth=mth["tmin_mth"][m0:m0 + g1 - g0], tmax_mth=mth["tmax_mth"][m0:m0 + g1 - g0])
                m0 += len(tile_days_mth(ctx[0], ctx[1], n, shape, g, out=out)["mth_groups"])
            else:
                tile_days(ctx[0], ctx[1], n, shape, out=out)
            d0 += n
        tile_end(ctx[0], ctx[1], shape, out=fin[months])
        e1.record(stream)
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1)

    one_pass(False)
    one_pass(True)
    ms = {False: [], True: []}
    for _ in range(args.reps):
        for m in (False, True):
            ms[m].append(one_pass(m))

    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        one_pass(True)
    kern = {"tile_month_kernel": [], "tile_apply_kernel": [], "tile_fix_kernel": []}
    for e in prof.events():
        for k in kern:
            if k in e.name and str(getattr(e, "device_type", "")).endswith("CUDA"):
                kern[k].append((e.time_range.start, e.time_range.elapsed_us() / 1e3))
    kern = {k: [d for _, d in sorted(v)] for k, v in kern.items()}

    # numpy on the host from the int16 record: what a reader of the daily files computes
    q = {k: dly[True][k].cpu().numpy() for k in ("tmin", "tmax")}
    st = fin[True]["status"].cpu().numpy()
    t = time.perf_counter()
    ref = {}
    for k in ("tmin", "tmax"):
        r = np.empty((start.size, T, T), np.float32)
        for g, (s, n) in enumerate(zip(start, ndays)):
            S = q[k][s:s + n].sum(axis=0, dtype=np.int32)
            r[g] = ((S / np.float64(n)) * np.float64(np.float32(0.01))).astype(np.float32)
        r[:, st != 0] = np.float32(9.969209968386869e+36)
        ref[k] = r
    host_s = time.perf_counter() - t
    equal_months = all(np.array_equal(mth[k + "_mth"].cpu().numpy().view(np.int32), ref[k].view(np.int32))
                       for k in ("tmin", "tmax"))
    equal_dailies = all(torch.equal(dly[False][k], dly[True][k]) for k in ("tmin", "tmax")) and \
        all(torch.equal(fin[False][k], fin[True][k]) for k in fin[False])

    rnd = lambda v: round(float(v), 4)
    mk_ms = kern["tile_month_kernel"]
    res = dict(
        tool="record_months", device=name, power_limit=power, tile_row0=int(r0), tile_col0=int(c0), cells=T * T,
        land_cells=int(land), nstns=args.nstns, year0=args.year0, years=args.years, ndays=nd, months=int(start.size),
        windows=len(yrs),
        stream_ms=dict(days=[rnd(x) for x in ms[False]], days_mth=[rnd(x) for x in ms[True]],
                       median_days=rnd(np.median(ms[False])), median_days_mth=rnd(np.median(ms[True]))),
        month_kernel_ms=dict(launches=len(mk_ms), total=rnd(sum(mk_ms)), per_window_mean=rnd(np.mean(mk_ms)),
                             per_window_min=rnd(min(mk_ms)), per_window_max=rnd(max(mk_ms)),
                             per_window=[rnd(x) for x in mk_ms]),
        window_kernels_ms_total=dict(apply=rnd(sum(kern["tile_apply_kernel"])), fix=rnd(sum(kern["tile_fix_kernel"]))),
        month_kernel_read_gb_per_year_window=rnd(2 * 365 * T * T * 2 / 1e9),
        numpy_host_s=rnd(host_s), numpy_values_read=int(2 * nd * T * T),
        equal_months_numpy=bool(equal_months), equal_dailies_with_without_months=bool(equal_dailies))
    print(json.dumps(res))
    if not (equal_months and equal_dailies and len(mk_ms) == len(yrs)):
        sys.exit(1)


if __name__ == "__main__":
    main()

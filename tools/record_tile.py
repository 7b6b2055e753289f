"""One full-land C5 tile (10 000-station table) over a multi-decade record, in year windows and in one whole-record call.

    python tools/record_tile.py [--year0 1948] [--years 68] [--nstns 10000]

The record is synthetic and seeded (synth.make_station_db over make_days(year0, years)).  Prints one JSON line:
  * device name and power limit (read-only nvidia-smi query);
  * year windows with device buffers: twxi_tile_begin, every twxi_tile_days and twxi_tile_end time (CUDA events on the
    contexts' stream, no host synchronisation in between) and the total;
  * the same with pinned host buffers, end to end (host clock around each call, which returns with the results in host
    memory);
  * twxi_interp_chunk on the same tile with device buffers;
  * cell-days/s for each (land cells x days / total time);
  * device memory each path's library calls need: torch.cuda.mem_get_info before and after the path's first (warm-up)
    pass, result buffers excluded.  The windowed path runs first, on fresh contexts, so its figure also holds the
    kNN / kriging workspaces that the whole-record call then reuses;
  * per-stage device times of a separate pass with stage timing on (begin: knn, nngh_params, krig, hat rows + state;
    windows: GWR apply and fixer / quantisation summed over the record; the whole-record call's five stages);
  * whether the windowed outputs (device and pinned) equal the whole-record outputs, byte for byte.
Every shape is warmed up before it is timed.  The obs tables (1 GB per variable for 68 years) exceed L2, so nothing timed
runs from a warm cache of the whole record.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np                                                              # noqa: E402

import bench                                                                    # noqa: E402
from topowx_b200 import db, synth, _lib                                         # noqa: E402
from topowx_b200.context import TwxiContext, interp_chunk, tile_begin, tile_days, tile_end    # noqa: E402


def gpu_name_power(dev):
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(dev)],
                           capture_output=True, text=True, timeout=60)
        name, power = [x.strip() for x in r.stdout.strip().split(",")[:2]]
        return name, power
    except Exception as e:                                                      # noqa: BLE001
        return "unknown (%s)" % e, "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--year0", type=int, default=1948)
    ap.add_argument("--years", type=int, default=68)
    ap.add_argument("--nstns", type=int, default=bench.NSTNS_C5)
    ap.add_argument("--device", type=int, default=0)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("record_tile.py measures on a CUDA device; none is available")
    torch.cuda.set_device(args.device)
    dev = torch.device("cuda", args.device)
    name, power = gpu_name_power(args.device)

    f, _, tiles, _ = bench.c5_tile_list(64)
    _, r0, c0, land = tiles[0]                                                  # the sample's largest land count
    days = synth.make_days(args.year0, args.years)
    nd = int(days.size)
    yrs = np.unique(days[db.YEAR], return_counts=True)[1].tolist()
    da = [synth.make_station_db(w, args.nstns, synth.conus_bbox(1.0), f, days, seed=synth.SEED_STNS) for w in (0, 1)]
    ctx = [TwxiContext(d, np.isnan(d.stns[db.BAD]), device=args.device) for d in da]
    del da
    wrk = torch.from_numpy(synth.make_wrk_chk_grid(f, r0, c0, bench.TILE, bench.TILE)).to(dev)
    T = bench.TILE
    shape = (T, T)
    stream = torch.cuda.current_stream(dev)
    lib = _lib.lib

    def ev():
        e = torch.cuda.Event(enable_timing=True)
        e.record(stream)
        return e

    def mk_fin():
        return dict(tmin_norm=torch.empty((12, T, T), dtype=torch.float32, device=dev),
                    tmax_norm=torch.empty((12, T, T), dtype=torch.float32, device=dev),
                    tmin_se=torch.empty((12, T, T), dtype=torch.float32, device=dev),
                    tmax_se=torch.empty((12, T, T), dtype=torch.float32, device=dev),
                    ninvalid=torch.empty((T, T), dtype=torch.int32, device=dev),
                    status=torch.empty((T, T), dtype=torch.uint8, device=dev))
    win = dict(tmin=torch.empty((nd, T, T), dtype=torch.int16, device=dev),
               tmax=torch.empty((nd, T, T), dtype=torch.int16, device=dev))
    win_fin = mk_fin()

    def windowed_device():
        e = [ev()]
        tile_begin(ctx[0], ctx[1], wrk)
        e.append(ev())
        d0 = 0
        for n in yrs:
            tile_days(ctx[0], ctx[1], n, shape, out=dict(tmin=win["tmin"][d0:d0 + n], tmax=win["tmax"][d0:d0 + n]))
            d0 += n
            e.append(ev())
        tile_end(ctx[0], ctx[1], shape, out=win_fin)
        e.append(ev())
        torch.cuda.synchronize(dev)
        ms = [a.elapsed_time(b) for a, b in zip(e[:-1], e[1:])]
        return dict(begin_ms=ms[0], window_ms=ms[1:-1], end_ms=ms[-1], total_ms=e[0].elapsed_time(e[-1]))

    def used():
        torch.cuda.synchronize(dev)
        fr, _ = torch.cuda.mem_get_info(dev)
        return fr

    # windowed path first, on fresh contexts: warm-up pass = memory measurement
    free0 = used()
    windowed_device()
    win_bytes = free0 - used()
    wd = windowed_device()

    whole = dict(tmin=torch.empty((nd, T, T), dtype=torch.int16, device=dev),
                 tmax=torch.empty((nd, T, T), dtype=torch.int16, device=dev), **mk_fin())
    free0 = used()
    interp_chunk(ctx[0], ctx[1], wrk, out=whole)
    whole_bytes = free0 - used()
    e0 = ev()
    interp_chunk(ctx[0], ctx[1], wrk, out=whole)
    e1 = ev()
    torch.cuda.synchronize(dev)
    whole_ms = e0.elapsed_time(e1)
    equal = all(torch.equal(win[k], whole[k]) for k in win) and all(torch.equal(win_fin[k], whole[k]) for k in win_fin)

    # pinned host buffers, end to end; each window is compared with the whole-record result outside the timed calls
    pin = dict(tmin=torch.empty((max(yrs), T, T), dtype=torch.int16).pin_memory(),
               tmax=torch.empty((max(yrs), T, T), dtype=torch.int16).pin_memory())
    pin_fin = {k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in mk_fin().items()}
    wrk_h = wrk.cpu().pin_memory()

    def windowed_pinned(check):
        ok = True
        t = time.perf_counter()
        tile_begin(ctx[0], ctx[1], wrk_h)
        torch.cuda.synchronize(dev)
        ms = [(time.perf_counter() - t) * 1e3]
        d0 = 0
        for n in yrs:
            t = time.perf_counter()
            o = tile_days(ctx[0], ctx[1], n, shape, out=dict(tmin=pin["tmin"][:n], tmax=pin["tmax"][:n]))
            ms.append((time.perf_counter() - t) * 1e3)
            if check:
                ok = ok and all(torch.equal(o[k], whole[k][d0:d0 + n].cpu()) for k in o)
            d0 += n
        t = time.perf_counter()
        tile_end(ctx[0], ctx[1], shape, out=pin_fin)
        ms.append((time.perf_counter() - t) * 1e3)
        if check:
            ok = ok and all(torch.equal(pin_fin[k], whole[k].cpu()) for k in pin_fin)
        return dict(begin_ms=ms[0], window_ms=ms[1:-1], end_ms=ms[-1], total_ms=float(sum(ms))), ok

    windowed_pinned(False)
    wp, equal_pinned = windowed_pinned(True)

    # per-stage device times, in a pass of their own (stage timing synchronises after every call)
    s5 = (C.c_float * 5)()
    lib.twxi_set_stage_timing(1)
    tile_begin(ctx[0], ctx[1], wrk)
    lib.twxi_get_stage_ms(s5)
    st_begin = [float(x) for x in s5]
    apply_ms = fix_ms = 0.0
    d0 = 0
    for n in yrs:
        tile_days(ctx[0], ctx[1], n, shape, out=dict(tmin=win["tmin"][d0:d0 + n], tmax=win["tmax"][d0:d0 + n]))
        d0 += n
        lib.twxi_get_stage_ms(s5)
        apply_ms += s5[3]
        fix_ms += s5[4]
    tile_end(ctx[0], ctx[1], shape, out=win_fin)
    interp_chunk(ctx[0], ctx[1], wrk, out=whole)
    torch.cuda.synchronize(dev)
    lib.twxi_get_stage_ms(s5)
    st_whole = [float(x) for x in s5]
    lib.twxi_set_stage_timing(0)

    cd = float(land) * nd
    rnd = lambda v: round(float(v), 3)
    for r in (wd, wp):
        r["window_ms_max"] = rnd(max(r["window_ms"]))
        r["window_ms_mean"] = rnd(np.mean(r["window_ms"]))
        r["window_ms"] = [rnd(x) for x in r["window_ms"]]
        r["begin_ms"], r["end_ms"], r["total_ms"] = rnd(r["begin_ms"]), rnd(r["end_ms"]), rnd(r["total_ms"])
        r["cell_days_per_s"] = float("%.4g" % (cd / (r["total_ms"] / 1e3)))
    wd["device_bytes"] = int(win_bytes)
    res = dict(
        tool="record_tile", device=name, power_limit=power, tile_row0=int(r0), tile_col0=int(c0), cells=T * T,
        land_cells=int(land), nstns=args.nstns, year0=args.year0, years=args.years, ndays=nd,
        windowed_device=wd, windowed_pinned=wp,
        whole_device=dict(total_ms=rnd(whole_ms), cell_days_per_s=float("%.4g" % (cd / (whole_ms / 1e3))),
                          device_bytes=int(whole_bytes)),
        windowed_over_whole=rnd(wd["total_ms"] / whole_ms),
        daily_buffer_bytes=dict(windowed=2 * T * T * (max(yrs) + 30) * 8, whole=2 * T * T * nd * 8),
        stage_ms=dict(begin=[rnd(x) for x in st_begin], windows_apply=rnd(apply_ms), windows_fixer=rnd(fix_ms),
                      whole=[rnd(x) for x in st_whole], order="knn, nngh_params, krig, gwr (hat rows | daily), "
                      "fixer_quantise (| state init)"),
        equal=bool(equal), equal_pinned=bool(equal_pinned))
    print(json.dumps(res))
    if not (equal and equal_pinned):
        sys.exit(1)


if __name__ == "__main__":
    main()

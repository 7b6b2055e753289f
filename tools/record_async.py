"""The record stream of one full-land C5 tile over 1948-2015 in year windows, synchronous against asynchronous.

    python tools/record_async.py [--year0 1948] [--years 68] [--nstns 10000] [--passes 3] [--trace out.json]

The tile, station table and record are those of tools/record_tile.py (row 250, col 3 500, 10 000 stations, seeded
synthetic record).  Prints one JSON line with the device name and power limit (read-only nvidia-smi query) and:
  * three paths, alternated over `--passes` passes after one warm-up pass each:
      device  device result buffers, synchronous calls (they only enqueue);
      pinned  pinned host buffers, synchronous calls (each returns with its results in host memory);
      async   pinned host buffers, twxi_tile_*_async into a ring of three result sets, then twxi_interp_chunk_wait;
    for each: device time (CUDA events on the contexts' stream from before the begin to after the end) and end-to-end
    time (host clock from the first submission to the last result byte in host memory);
  * four tiles back to back, pinned buffers, synchronous against asynchronous (each tile's begin submitted right after
    the previous tile's end), end to end;
  * the device -> host copy time of one year window alone (both variables, device buffer to pinned buffer);
  * byte identity: every window and end output of `pinned` and `async` against `device` (one pass each, outside the
    timed passes), and CRC-32s of every output of the four-tile legs, synchronous against asynchronous;
  * with --trace: one torch.profiler pass of its own (CUDA activities) over the begin and the first windows of the async
    path, written to that file, and from it the share of device -> host copy time that runs while a tile_apply_kernel or
    tile_fix_kernel of a later window runs.
"""
import argparse
import json
import os
import sys
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np                                                              # noqa: E402

import bench                                                                    # noqa: E402
from record_tile import gpu_name_power                                          # noqa: E402
from topowx_b200 import db, synth                                               # noqa: E402
from topowx_b200.context import (TwxiContext, interp_chunk_wait, tile_begin, tile_days, tile_end)   # noqa: E402

FIN = ("tmin_norm", "tmax_norm", "tmin_se", "tmax_se", "ninvalid", "status")


def overlap_from_trace(path):
    """Device -> host copy time inside the trace, and the part of it that overlaps a window kernel (tile_apply_kernel /
    tile_fix_kernel) on another stream."""
    with open(path) as fh:
        ev = json.load(fh).get("traceEvents", [])
    copies = [e for e in ev if e.get("cat") == "gpu_memcpy" and "DtoH" in e.get("name", "")]
    kern = [e for e in ev if e.get("cat") == "kernel" and ("tile_apply_kernel" in e.get("name", "")
                                                           or "tile_fix_kernel" in e.get("name", ""))]
    ks = sorted((float(k["ts"]), float(k["ts"]) + float(k["dur"]), k.get("args", {}).get("stream")) for k in kern)
    tot = ov = 0.0
    for c in copies:
        a, b = float(c["ts"]), float(c["ts"]) + float(c["dur"])
        s = c.get("args", {}).get("stream")
        tot += b - a
        # kernels on the compute stream never overlap each other, so the intersections add up
        ov += sum(max(0.0, min(b, k1) - max(a, k0)) for k0, k1, ks_ in ks if ks_ != s)
    return dict(dtoh_copies=len(copies), window_kernels=len(kern), dtoh_us=round(tot, 1), dtoh_overlapped_us=round(ov, 1),
                overlapped_share=round(ov / tot, 3) if tot else None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--year0", type=int, default=1948)
    ap.add_argument("--years", type=int, default=68)
    ap.add_argument("--nstns", type=int, default=bench.NSTNS_C5)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--passes", type=int, default=3)
    ap.add_argument("--tiles", type=int, default=4, help="tiles of the back-to-back leg")
    ap.add_argument("--trace", default=None, help="write a torch.profiler trace of the async path here")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("record_async.py measures on a CUDA device; none is available")
    torch.cuda.set_device(args.device)
    dev = torch.device("cuda", args.device)
    name, power = gpu_name_power(args.device)

    f, _, tiles, _ = bench.c5_tile_list(64)
    days = synth.make_days(args.year0, args.years)
    nd = int(days.size)
    yrs = np.unique(days[db.YEAR], return_counts=True)[1].tolist()
    da = [synth.make_station_db(w, args.nstns, synth.conus_bbox(1.0), f, days, seed=synth.SEED_STNS) for w in (0, 1)]
    ctx = [TwxiContext(d, np.isnan(d.stns[db.BAD]), device=args.device) for d in da]
    del da
    T = bench.TILE
    shape = (T, T)
    wrks = [torch.from_numpy(synth.make_wrk_chk_grid(f, r0, c0, T, T)).pin_memory() for _, r0, c0, _ in
            tiles[:max(args.tiles, 1)]]
    _, r0, c0, land = tiles[0]                                                   # the sample's largest land count
    wrk_d = wrks[0].to(dev)
    stream = torch.cuda.current_stream(dev)
    pin = lambda shp, dt: torch.empty(shp, dtype=dt).pin_memory()

    def ev():
        e = torch.cuda.Event(enable_timing=True)
        e.record(stream)
        return e

    def fin_set(mk):
        return dict(tmin_norm=mk((12, T, T), torch.float32), tmax_norm=mk((12, T, T), torch.float32),
                    tmin_se=mk((12, T, T), torch.float32), tmax_se=mk((12, T, T), torch.float32),
                    ninvalid=mk((T, T), torch.int32), status=mk((T, T), torch.uint8))
    dmk = lambda shp, dt: torch.empty(shp, dtype=dt, device=dev)
    win_d = dict(tmin=dmk((nd, T, T), torch.int16), tmax=dmk((nd, T, T), torch.int16))
    fin_d = fin_set(dmk)
    sets = [dict(tmin=pin((max(yrs), T, T), torch.int16), tmax=pin((max(yrs), T, T), torch.int16)) for _ in range(3)]
    fins = [fin_set(pin) for _ in range(3)]

    def run_device():
        t = time.perf_counter()
        e0 = ev()
        tile_begin(ctx[0], ctx[1], wrk_d)
        d0 = 0
        for n in yrs:
            tile_days(ctx[0], ctx[1], n, shape, out=dict(tmin=win_d["tmin"][d0:d0 + n], tmax=win_d["tmax"][d0:d0 + n]))
            d0 += n
        tile_end(ctx[0], ctx[1], shape, out=fin_d)
        e1 = ev()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1), (time.perf_counter() - t) * 1e3, True

    def run_pinned(wrk, check=False, crc=None):
        ok = True
        t = time.perf_counter()
        e0 = ev()
        tile_begin(ctx[0], ctx[1], wrk)
        d0 = 0
        for n in yrs:
            o = tile_days(ctx[0], ctx[1], n, shape, out={k: v[:n] for k, v in sets[0].items()})
            if check:
                ok = ok and all(torch.equal(o[k], win_d[k][d0:d0 + n].cpu()) for k in o)
            if crc is not None:
                crc.append([zlib.crc32(o[k].numpy()) for k in ("tmin", "tmax")])
            d0 += n
        tile_end(ctx[0], ctx[1], shape, out=fins[0])
        e1 = ev()
        ms = (time.perf_counter() - t) * 1e3
        torch.cuda.synchronize(dev)
        if check:
            ok = ok and all(torch.equal(fins[0][k], fin_d[k].cpu()) for k in FIN)
        if crc is not None:
            crc.append([zlib.crc32(fins[0][k].numpy()) for k in FIN])
        return e0.elapsed_time(e1), ms, ok

    def run_async(wrk_list, check=False, crc=None, nwin=None):
        """Every tile of wrk_list back to back, all calls asynchronous; window t's set is examined (check / crc) once
        t+2 has been submitted, the last ones after the wait."""
        ok = True
        held = []                                                   # (kind, buffers, first day, days) per submission

        def examine(item):
            nonlocal ok
            kind, o, d0, n = item
            if kind == "win":
                if check:
                    ok = ok and all(torch.equal(o[k], win_d[k][d0:d0 + n].cpu()) for k in o)
                if crc is not None:
                    crc.append([zlib.crc32(o[k].numpy()) for k in ("tmin", "tmax")])
            elif kind == "fin":
                if check:
                    ok = ok and all(torch.equal(o[k], fin_d[k].cpu()) for k in FIN)
                if crc is not None:
                    crc.append([zlib.crc32(o[k].numpy()) for k in FIN])

        def submitted(item):
            held.append(item)
            if len(held) > 2:
                examine(held.pop(0))
        t = time.perf_counter()
        e0 = ev()
        k = 0
        for wrk in wrk_list:
            tile_begin(ctx[0], ctx[1], wrk, wait=False)
            submitted(("begin", None, 0, 0))
            d0 = 0
            for n in (yrs if nwin is None else yrs[:nwin]):
                o = tile_days(ctx[0], ctx[1], n, shape, out={key: v[:n] for key, v in sets[k % 3].items()}, wait=False)
                k += 1
                submitted(("win", o, d0, n))
                d0 += n
            if nwin is not None:
                break
            o = tile_end(ctx[0], ctx[1], shape, out=fins[k % 3], wait=False)
            k += 1
            submitted(("fin", o, 0, 0))
        interp_chunk_wait(ctx[0], host_sync=False)                  # orders the stream after the last copy
        e1 = ev()
        interp_chunk_wait(ctx[0])
        ms = (time.perf_counter() - t) * 1e3
        for item in held:
            examine(item)
        return e0.elapsed_time(e1), ms, ok

    # warm-up of every path = byte checks (outside the timed passes)
    run_device()
    _, _, eq_pinned = run_pinned(wrks[0], check=True)
    _, _, eq_async = run_async(wrks[:1], check=True)
    res_ms = {p: [] for p in ("device", "pinned", "async")}
    for _ in range(args.passes):
        for p, fn in (("device", run_device), ("pinned", lambda: run_pinned(wrks[0])),
                      ("async", lambda: run_async(wrks[:1]))):
            dms, ems, _ = fn()
            res_ms[p].append((dms, ems))

    # four tiles back to back
    crc_s, crc_a = [], []
    for w in wrks:
        run_pinned(w, crc=crc_s)
    run_async(wrks, crc=crc_a)
    multi = {"sync": [], "async": []}
    for _ in range(args.passes):
        t = time.perf_counter()
        for w in wrks:
            run_pinned(w)
        multi["sync"].append((time.perf_counter() - t) * 1e3)
        multi["async"].append(run_async(wrks)[1])

    # the device -> host copy of one year window alone
    n = max(yrs)
    src = dmk((2, n, T, T), torch.int16)
    dst = pin((2, n, T, T), torch.int16)
    dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize(dev)
    cms = []
    for _ in range(5):
        e0 = ev()
        dst.copy_(src, non_blocking=True)
        e1 = ev()
        torch.cuda.synchronize(dev)
        cms.append(e0.elapsed_time(e1))
    copy_bytes = 2 * n * T * T * 2

    trace = None
    if args.trace:
        from torch.profiler import profile, ProfilerActivity
        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            run_async(wrks[:1], nwin=6)
        prof.export_chrome_trace(args.trace)
        trace = dict(file=os.path.basename(args.trace), windows=6, **overlap_from_trace(args.trace))

    cd = float(land) * nd
    rnd = lambda v: round(float(v), 3)

    def summ(v):
        d = np.array([x[0] for x in v]); e = np.array([x[1] for x in v])
        return dict(device_ms=[rnd(x) for x in d], end_to_end_ms=[rnd(x) for x in e],
                    end_to_end_ms_median=rnd(np.median(e)), per_window_ms=rnd(np.median(e) / len(yrs)),
                    cell_days_per_s=float("%.4g" % (cd / (np.median(e) / 1e3))))
    res = dict(
        tool="record_async", device=name, power_limit=power, tile_row0=int(r0), tile_col0=int(c0), cells=T * T,
        land_cells=int(land), nstns=args.nstns, year0=args.year0, years=args.years, ndays=nd, windows=len(yrs),
        paths={p: summ(v) for p, v in res_ms.items()},
        back_to_back=dict(tiles=len(wrks), sync_ms=[rnd(x) for x in multi["sync"]],
                          async_ms=[rnd(x) for x in multi["async"]], sync_ms_median=rnd(np.median(multi["sync"])),
                          async_ms_median=rnd(np.median(multi["async"]))),
        window_copy=dict(bytes=copy_bytes, ms=rnd(np.median(cms)), gb_per_s=rnd(copy_bytes / np.median(cms) / 1e6)),
        equal_pinned=bool(eq_pinned), equal_async=bool(eq_async), back_to_back_equal=bool(crc_s == crc_a),
        trace=trace)
    print(json.dumps(res))
    if not (eq_pinned and eq_async and crc_s == crc_a):
        sys.exit(1)


if __name__ == "__main__":
    main()

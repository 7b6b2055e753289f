#!/usr/bin/env python
'''
Gridded interpolation driver: the Python-3 / GPU counterpart of scripts/step25_mpi_interp_tair.py.

    python scripts/step25_interp_tair.py --out /tmp/twx_out [--rows 500 --cols 750] [--format nc|raw]
                                         [--year0 1948 --years 68 --window year] [--months]
    torchrun --nproc-per-node N scripts/step25_interp_tair.py ...     (one process per GPU)

The reference runs an MPI task farm: rank 0 reads every 50x50 work chunk's 27 predictor windows from netCDF and hands it
to a worker (step25:266-314), the workers loop over the cells (step25:96-198), rank 1 writes netCDF tiles (step25:200-264).
Here every rank builds the same ordered tile list with Tiler over the predictor rasters on disk (PredictorStore), takes its
share with partition_chunks (whole tiles, greedy by unmasked cells; stations replicated on every GPU, no collective), a
background thread reads each tile's windows once into pinned memory (TileFeed), the tile goes through
PtInterpTair.interp_chunk(wait=False) = twxi_interp_chunk_async with three sets of pinned result buffers in flight, and a
writer pool writes the reference's netCDF tiles (TileWriter; raw .npy with --format raw).  Without rasters at --rasters a
synthetic window of the CONUS grid is generated first (topowx_b200.synth).
The synthetic station record covers --years calendar years from --year0.  --window record (default) computes each tile's
whole record in one call; --window year goes through PtInterpTair.interp_chunk_stream instead: kriging and GWR hat rows
once per tile, then one calendar year at a time, so a multi-decade record never sits whole on the device or in pinned
memory.  Each year is written as it comes (TileWriter.open_tile_stream; --format raw: one .npy per year window).  The year
windows are pipelined: every call is submitted without waiting (interp_chunk_stream(wait=False)) into a ring of pinned
result sets, so a window's device -> host copy overlaps the next window's kernels and the next tile's kriging overlaps
this tile's last copies; writer threads take each set once the library's ownership rule releases it.
--months also writes the monthly means of the dailies beside the daily tiles (<tile>_<var>_mthly.nc through
TileWriter.open_tile_stream_mthly; --format raw: one <tile>_<var>_mthly_<day0>.npy per window and variable).  It always
goes through interp_chunk_stream(months=True); with --window record the stream has one window covering the whole record,
which gives the bytes of the whole-record call.
'''
import argparse
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from topowx_b200 import synth                                     # noqa: E402
from topowx_b200.interp import (PtInterpTair, Tiler, partition_chunks, PredictorStore, TileFeed,     # noqa: E402
                                AsyncTileWriter, TileWriter)

P_TILESIZE = 250                                                  # step25_mpi_interp_tair.py:349-352


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="/tmp/twx_tiles")
    ap.add_argument("--rasters", default=None, help="PredictorStore directory (created with synthetic rasters if missing)")
    ap.add_argument("--row0", type=int, default=synth.TILE_ROW0)
    ap.add_argument("--col0", type=int, default=synth.TILE_COL0)
    ap.add_argument("--rows", type=int, default=P_TILESIZE)
    ap.add_argument("--cols", type=int, default=2 * P_TILESIZE)
    ap.add_argument("--nstns", type=int, default=4000)
    ap.add_argument("--format", default="nc", choices=["nc", "raw"])
    ap.add_argument("--year0", type=int, default=1995, help="first year of the synthetic station record")
    ap.add_argument("--years", type=int, default=1, help="calendar years of the synthetic station record")
    ap.add_argument("--window", default="record", choices=["record", "year"],
                    help="whole record per tile in one call, or one calendar year at a time")
    ap.add_argument("--months", action="store_true", help="also write the monthly means of the dailies")
    args = ap.parse_args()
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)

    f = synth.Fields()
    days = synth.make_days(args.year0, args.years)
    rpath = args.rasters or os.path.join(args.out, "rasters")
    if not os.path.exists(os.path.join(rpath, "mask.npy")):
        if rank == 0:
            PredictorStore.create_synthetic(rpath, f, args.row0, args.col0, args.rows, args.cols)
        while not os.path.exists(os.path.join(rpath, "mask.npy")):
            time.sleep(0.2)
        time.sleep(0.5 if rank else 0.0)
    store = PredictorStore(rpath)
    tiler = Tiler(store, store.attrs(), P_TILESIZE, P_TILESIZE, P_TILESIZE, P_TILESIZE)     # one work chunk per tile
    info = tiler.build_tile_grid_info()
    lat, lon = store.variables["lat"], store.variables["lon"]
    bbox = (float(lat.min()) - 4.0, float(lat.max()) + 4.0, float(lon.min()) - 4.0, float(lon.max()) + 4.0)
    da = [synth.make_station_db(w, args.nstns, bbox, f, days) for w in (0, 1)]
    pt_interp = PtInterpTair(da[0], da[1], device=local_rank)

    mine = partition_chunks(tiler.tile_chks, tiler.mask, P_TILESIZE, P_TILESIZE, world, rank)
    nd = days.size
    if args.window == "year":
        return pipelined(args, pt_interp, TileFeed(tiler, chunks=mine, depth=4), TileWriter(info, args.out), days, rank,
                         world, len(mine))
    if args.months:
        return streamed(args, pt_interp, TileFeed(tiler, chunks=mine, depth=4), TileWriter(info, args.out), days, rank, world,
                       len(mine))
    pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()
    outs = [dict(tmin=pin((nd, P_TILESIZE, P_TILESIZE), torch.int16), tmax=pin((nd, P_TILESIZE, P_TILESIZE), torch.int16),
                 tmin_norm=pin((12, P_TILESIZE, P_TILESIZE), torch.float32), tmax_norm=pin((12, P_TILESIZE, P_TILESIZE), torch.float32),
                 tmin_se=pin((12, P_TILESIZE, P_TILESIZE), torch.float32), tmax_se=pin((12, P_TILESIZE, P_TILESIZE), torch.float32),
                 ninvalid=pin((P_TILESIZE, P_TILESIZE), torch.int32), status=pin((P_TILESIZE, P_TILESIZE), torch.uint8))
            for _ in range(3)]
    writer = AsyncTileWriter(info, args.out, days, fmt=args.format, nthreads=3)
    feed = TileFeed(tiler, chunks=mine, depth=4)
    t0 = time.time()
    pend, ncells = [], 0

    def retire(j):
        nonlocal ncells
        tid, slot = pend[j]
        o = {k: v.numpy() for k, v in outs[slot].items()}
        ncells += int((o["status"] == 0).sum())
        writer.submit(tid, o, copy=True)                        # copied: the pinned set is reused two submissions later

    for t, (k, tid, wrk) in enumerate(feed):
        pt_interp.interp_chunk(wrk, out=outs[t % 3], wait=False)
        pend.append((tid, t % 3))
        if t >= 2:                                              # tile t-2 is complete once tile t has been submitted
            retire(t - 2)
    pt_interp.interp_chunk_wait()
    for j in range(max(len(pend) - 2, 0), len(pend)):
        retire(j)
    nbytes = writer.wait()
    writer.close()
    dt = time.time() - t0
    print("rank %d/%d: %d tiles, %d cells x %d days in %.2f s = %.3g cell-days/s from rasters on disk (%.1f MB read) to %s "
          "tiles on disk (%.1f MB)" % (rank, world, len(mine), ncells, nd, dt, ncells * nd / max(dt, 1e-9),
                                       feed.bytes_read / 1e6, writer.tw.format if args.format == "nc" else "raw .npy",
                                       nbytes / 1e6))


N_SETS = 5       # pinned result sets: three the library may own (submissions t, t+1, t+2), two with the writers


def pipelined(args, pt_interp, feed, tw, days, rank, world, ntiles):
    '''
    --window year: every begin, year window and end is submitted without waiting (interp_chunk_stream(wait=False)), into
    a ring of pinned result sets sized for the longest window.  A submission's set is handed to the writers once two
    further submissions have been made (the library's ownership rule) or after the final wait, and goes back to the ring
    when its writes finish.  The device -> host copy of a window overlaps the kernels of the next one, and the next tile's
    begin is submitted right after this tile's end.  The files are those of the synchronous loop, byte for byte.
    '''
    import collections
    import queue
    from concurrent.futures import ThreadPoolExecutor
    import torch
    from topowx_b200.db import month_runs
    nc = args.format == "nc"
    T = P_TILESIZE
    yrs = np.unique(days["YEAR"], return_counts=True)[1].tolist()
    start, mlen, _, _ = month_runs(days)
    ends, bounds = start + mlen, np.cumsum([0] + yrs)
    max_mth = int(max(np.searchsorted(ends, b, side="right") - np.searchsorted(ends, a, side="right")
                      for a, b in zip(bounds[:-1], bounds[1:])))
    pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()
    ring = queue.Queue()
    for _ in range(N_SETS):
        st = dict(tmin=pin((max(yrs), T, T), torch.int16), tmax=pin((max(yrs), T, T), torch.int16),
                  tmin_norm=pin((12, T, T), torch.float32), tmax_norm=pin((12, T, T), torch.float32),
                  tmin_se=pin((12, T, T), torch.float32), tmax_se=pin((12, T, T), torch.float32),
                  ninvalid=pin((T, T), torch.int32), status=pin((T, T), torch.uint8))
        if args.months:
            st.update(tmin_mth=pin((max_mth, T, T), torch.float32), tmax_mth=pin((max_mth, T, T), torch.float32))
        ring.put(st)
    # netCDF libraries are not thread-safe: one writer thread does every netCDF call, in submission order
    pool = ThreadPoolExecutor(max_workers=1 if nc else 3)
    futures, owned = [], collections.deque()      # owned: submissions whose buffers the library may still write

    def hand(item):
        if item is not None:
            job, st = item

            def run():
                try:
                    return job()
                finally:
                    ring.put(st)
            futures.append(pool.submit(run))

    def submitted(item):
        owned.append(item)
        if len(owned) > 2:                                      # submission t is complete once t+2 has been submitted
            hand(owned.popleft())

    def write_window(tid, h, d0, m0, o):
        n = 0
        for v in ("tmin", "tmax"):
            q = o[v].numpy()
            if nc:
                h["days"][v].write_days(d0, q)
            else:
                np.save(os.path.join(args.out, tid, "%s_%s_%05d.npy" % (tid, v, d0)), q)
                n += q.nbytes
            if args.months:
                m = o[v + "_mth"].numpy()
                if nc:
                    h["mth"][v].write_months(m0, m)
                else:
                    np.save(os.path.join(args.out, tid, "%s_%s_mthly_%05d.npy" % (tid, v, d0)), m)
                    n += m.nbytes
        return n, 0

    def write_end(tid, h, fin):
        fin = {k: a.numpy() for k, a in fin.items()}
        n = 0
        for v in ("tmin", "tmax"):
            if nc:
                h["days"][v].close(fin[v + "_norm"], fin[v + "_se"], fin["ninvalid"])
                n += os.path.getsize(tw._fpath(tid, v))
                if args.months:
                    h["mth"][v].close()
                    n += os.path.getsize(tw._fpath_mthly(tid, v))
        if not nc:
            for key, a in fin.items():
                np.save(os.path.join(args.out, tid, "%s_%s.npy" % (tid, key)), a)
                n += a.nbytes
        return n, int((fin["status"] == 0).sum())

    def open_tile(tid, h):
        h["days"] = {v: tw.open_tile_stream(tid, v, days) for v in ("tmin", "tmax")}
        if args.months:
            h["mth"] = {v: tw.open_tile_stream_mthly(tid, v, days) for v in ("tmin", "tmax")}
        return 0, 0

    fin_keys = ("tmin_norm", "tmax_norm", "tmin_se", "tmax_se", "ninvalid", "status")
    t0 = time.time()                                            # after the ring, as the feed's buffers are set up before
    for k, tid, wrk in feed:
        s = pt_interp.interp_chunk_stream(wrk, months=args.months, wait=False)
        submitted(None)                                         # the begin: wrk is the library's until t+2
        os.makedirs(os.path.join(args.out, tid), exist_ok=True)
        h = {}
        if nc:
            futures.append(pool.submit(open_tile, tid, h))
        m0 = 0
        for n in yrs:
            st = ring.get()
            out = dict(tmin=st["tmin"][:n], tmax=st["tmax"][:n])
            if args.months:
                g0, g1 = s.groups.completed(n)
                out.update(tmin_mth=st["tmin_mth"][:g1 - g0], tmax_mth=st["tmax_mth"][:g1 - g0])
            d0 = s.day0
            o = s.days(n, out=out)
            submitted((lambda tid=tid, h=h, d0=d0, m0=m0, o=o: write_window(tid, h, d0, m0, o), st))
            m0 += len(o.get("mth_groups", ()))
        st = ring.get()
        fin = s.finish(out={key: st[key] for key in fin_keys})
        submitted((lambda tid=tid, h=h, fin=fin: write_end(tid, h, fin), st))
    pt_interp.interp_chunk_wait()
    while owned:
        hand(owned.popleft())
    ncells, nbytes = 0, 0
    for f in futures:
        n, c = f.result()
        nbytes += n
        ncells += c
    pool.shutdown()
    dt = time.time() - t0
    print("rank %d/%d: %d tiles, %d cells x %d days in %.2f s = %.3g cell-days/s in year windows, pipelined%s to %s "
          "tiles on disk (%.1f MB)" % (rank, world, ntiles, ncells, days.size, dt, ncells * days.size / max(dt, 1e-9),
                                       " with monthly means" if args.months else "",
                                       tw.format if nc else "raw .npy", nbytes / 1e6))


def streamed(args, pt_interp, feed, tw, days, rank, world, ntiles):
    '''--window record --months: one window covering each tile's whole record, written as the synchronous call returns.'''
    t0 = time.time()
    ncells, nbytes = 0, 0
    for k, tid, wrk in feed:
        s = pt_interp.interp_chunk_stream(wrk, months=args.months)
        d = os.path.join(args.out, tid)
        os.makedirs(d, exist_ok=True)
        nc = args.format == "nc"
        hs = {v: tw.open_tile_stream(tid, v, days) for v in ("tmin", "tmax")} if nc else None
        hm = {v: tw.open_tile_stream_mthly(tid, v, days) for v in ("tmin", "tmax")} if nc and args.months else None
        windows = iter([(0, s.days(days.size))])
        m0 = 0
        for d0, o in windows:
            for v in ("tmin", "tmax"):
                if hs:
                    hs[v].write_days(d0, o[v])
                else:
                    np.save(os.path.join(d, "%s_%s_%05d.npy" % (tid, v, d0)), o[v])
                    nbytes += o[v].nbytes
                if hm:
                    hm[v].write_months(m0, o[v + "_mth"])
                elif args.months:
                    np.save(os.path.join(d, "%s_%s_mthly_%05d.npy" % (tid, v, d0)), o[v + "_mth"])
                    nbytes += o[v + "_mth"].nbytes
            if args.months:
                m0 += len(o["mth_groups"])
        fin = s.finish()
        for v in ("tmin", "tmax"):
            if hs:
                hs[v].close(fin[v + "_norm"], fin[v + "_se"], fin["ninvalid"])
                nbytes += os.path.getsize(tw._fpath(tid, v))
            if hm:
                hm[v].close()
                nbytes += os.path.getsize(tw._fpath_mthly(tid, v))
        if not hs:
            for key, a in fin.items():
                np.save(os.path.join(d, "%s_%s.npy" % (tid, key)), a)
                nbytes += a.nbytes
        ncells += int((fin["status"] == 0).sum())
    dt = time.time() - t0
    print("rank %d/%d: %d tiles, %d cells x %d days in %.2f s = %.3g cell-days/s in %s windows%s to %s tiles on disk "
          "(%.1f MB)" % (rank, world, ntiles, ncells, days.size, dt, ncells * days.size / max(dt, 1e-9), args.window,
                         " with monthly means" if args.months else "", tw.format if args.format == "nc" else "raw .npy",
                         nbytes / 1e6))


if __name__ == "__main__":
    main()

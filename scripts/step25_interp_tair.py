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
memory.  Each year is written as it comes (TileWriter.open_tile_stream; --format raw: one .npy per year window).
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
    if args.window == "year" or args.months:
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


def streamed(args, pt_interp, feed, tw, days, rank, world, ntiles):
    t0 = time.time()
    ncells, nbytes = 0, 0
    for k, tid, wrk in feed:
        s = pt_interp.interp_chunk_stream(wrk, months=args.months)
        d = os.path.join(args.out, tid)
        os.makedirs(d, exist_ok=True)
        nc = args.format == "nc"
        hs = {v: tw.open_tile_stream(tid, v, days) for v in ("tmin", "tmax")} if nc else None
        hm = {v: tw.open_tile_stream_mthly(tid, v, days) for v in ("tmin", "tmax")} if nc and args.months else None
        windows = s.years() if args.window == "year" else iter([(0, s.days(days.size))])
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

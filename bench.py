#!/usr/bin/env python
"""Benchmark of the TopoWx interpolation hot path (BASELINE.json metric: interpolated cell-days/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload = BASELINE.json configs[4] (C5): the CONUS 30-arcsec grid (3250 x 7000 cells, synthetic land mask, ~56 % land),
10 000 synthetic stations per variable, one year (365 days) of daily Tmin+Tmax (12 monthly-normal regression krigings +
daily-anomaly GWR per variable, Tmin>=Tmax fixer, int16 quantisation).  A step = ONE PASS OVER A FIXED LIST OF DISTINCT
TILES taken from the reference's ordered tile list (Tiler.tile_chks, twx/interp/tiling.py:131-165): by default a declared
sample of 64 of the 255 tiles that contain land, evenly spaced over the list (TWX_BENCH_TILES=all runs every tile).  With
--gpus N (torchrun) the SAME list is divided among the N ranks (strong scaling): ranks pull tiles, largest first, from a
shared counter the way the reference's workers pull chunks from the coordinator rank
(scripts/step25_mpi_interp_tair.py:293-305); stations are replicated, there is no collective on the data path.
Prints ONE JSON line on rank 0; secondary figures (configs[1] tile, C3 leave-one-out, C4 normals only) ride in the same line.
--dump-outputs DIR writes what the last timed step computed, for comparing two builds output for output (OutputDump).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "interpolated cell-days/sec (daily Tmin+Tmax, 30\" grid)"
UNIT = "cell-days/s"
NSTNS = 2000                 # configs[1]
NSTNS_C5 = 10000
TILE = 250
NDAYS = 365
NTILES_DEFAULT = 64


# ---- inputs ----------------------------------------------------------------------------------------------------------
def build_inputs(rank):
    """configs[1]: the interior benchmark tile with ~2000 stations per variable (secondary line, tools/)."""
    from topowx_b200 import synth
    f = synth.Fields()
    days = synth.make_days(1995, 1)
    del rank
    col0 = synth.TILE_COL0
    bbox = synth.tile_bbox(col0=col0)
    da = [synth.make_station_db(w, NSTNS, bbox, f, days, seed=synth.SEED_STNS) for w in (0, 1)]
    wrk = synth.make_wrk_chk(f, synth.TILE_ROW0, col0, TILE, TILE)
    return da, wrk


def conus_mask(f):
    from topowx_b200 import synth
    lat = synth.grid_lats(np.arange(synth.GRID_NROWS))
    lon = synth.grid_lons(np.arange(synth.GRID_NCOLS))
    mask = np.zeros((synth.GRID_NROWS, synth.GRID_NCOLS), dtype=bool)
    for r0 in range(0, synth.GRID_NROWS, TILE):
        mask[r0:r0 + TILE] = synth.make_wrk_chk_grid_mask(f, r0, 0, TILE, synth.GRID_NCOLS)
    return mask, lat, lon


def c5_tile_list(ntiles):
    """(fields, tiler, tiles): tiles = [(tile number, row0, col0, land cells)] of the declared sample, in the order they
    are handed out (largest first)."""
    from topowx_b200 import synth
    from topowx_b200.interp.tiling import Tiler
    f = synth.Fields()
    mask, lat, lon = conus_mask(f)
    tiler = Tiler(dict(mask=mask, lon=lon, lat=lat), [], TILE, TILE, TILE, TILE)     # one work chunk per tile
    chks = tiler.tile_chks                                                           # reference order, land tiles only
    if ntiles is None or ntiles >= len(chks):
        sel = list(range(len(chks)))
    else:
        sel = sorted(set(np.linspace(0, len(chks) - 1, ntiles).astype(int).tolist()))
    tiles = []
    for i in sel:
        k, r0, c0, _, _ = chks[i]
        tiles.append((int(k), int(r0), int(c0), int(mask[r0:r0 + TILE, c0:c0 + TILE].sum())))
    tiles.sort(key=lambda t: (-t[3], t[0]))
    return f, tiler, tiles, len(chks)


def c5_stations(f):
    from topowx_b200 import synth
    days = synth.make_days(1995, 1)
    return [synth.make_station_db(w, NSTNS_C5, synth.conus_bbox(1.0), f, days, seed=synth.SEED_STNS) for w in (0, 1)]


def ked_flops(kn):
    """Algorithmic FLOPs of the kriging stage (SURVEY §8d F_ked with pair distances looked up, c_exp = 20):
    n^3/3 + 2n^2(p+2) + (n^2/2 + n)*20 + 2np^2 + p^3/3 + 4np per (cell, month, variable), p = 5."""
    n = kn.astype(np.float64)
    p = 5.0
    return float(np.sum(n ** 3 / 3 + 2 * n * n * (p + 2) + (n * n / 2 + n) * 20 + 2 * n * p * p + p ** 3 / 3 + 4 * n * p))


def gwr_flops(ka, days_in_month):
    """SURVEY §8d: F_gwr = 2kq^2 + q^3/3 + 2q^2 + 2kq (hat row, q = 6) + F_app = 2kD per (cell, month, variable)."""
    k = ka.astype(np.float64)
    q = 6.0
    D = np.asarray(days_in_month, dtype=np.float64)[None, :]
    return float(np.sum(2 * k * q * q + q ** 3 / 3 + 2 * q * q + 2 * k * q + 2 * k * D))


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        threading.Thread.__init__(self, daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
                if self.stop_flag:
                    break
        except Exception:
            pass

    def stop(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower() == "active"})
        busy = [s for s in sm if s > 0.5 * (max(mx) if mx else 1)] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


DUMP_BYTES = 64 * 10 ** 6
DUMP_SEED = 2024


class OutputDump(object):
    """--dump-outputs: what twxi_interp_chunk returned for every tile of the last timed step, at a fixed seeded sample of
    cells (the same row-major cell indices in every tile; as many as fit DUMP_BYTES).  Gathered on the stream right after
    each tile, before its result buffers are reused.  Files: <key>.npy of shape (tiles in list order, ..., cells), the
    int16 / uint8 results as float32 and ninvalid as float64 (exact)."""
    KEYS = ("tmin", "tmax", "tmin_norm", "tmax_norm", "tmin_se", "tmax_se", "ninvalid", "status")

    def __init__(self, ntiles):
        import torch
        per_cell = (2 * NDAYS + 4 * 12 + 1) * 4 + 8
        n = min(TILE * TILE, (DUMP_BYTES - len(self.KEYS) * 4096) // (ntiles * per_cell))
        cells = np.sort(np.random.default_rng(DUMP_SEED).choice(TILE * TILE, n, replace=False))
        self.cells = torch.from_numpy(cells).cuda()
        lead = dict(tmin=(NDAYS,), tmax=(NDAYS,), ninvalid=(), status=())
        self.buf = {k: torch.zeros((ntiles,) + lead.get(k, (12,)) + (n,), device="cuda",
                                   dtype=torch.float64 if k == "ninvalid" else torch.float32) for k in self.KEYS}

    def take(self, i, out):
        for k, b in self.buf.items():
            v = out[k]
            b[i] = v.reshape(v.shape[:-2] + (-1,)).index_select(-1, self.cells)

    def save(self, path, world, rank):
        """Every rank holds the tiles it pulled (zeros elsewhere): a sum over ranks assembles the whole list exactly."""
        import torch.distributed as dist
        if world > 1:
            for b in self.buf.values():
                dist.all_reduce(b)
        if rank == 0:
            os.makedirs(path, exist_ok=True)
            for k, b in self.buf.items():
                np.save(os.path.join(path, k + ".npy"), b.cpu().numpy())


def sample_cells(wrk, n, seed=7):
    r = np.random.default_rng(seed)
    land = np.nonzero(wrk[2].ravel() != 0)[0]
    flat = r.choice(land, size=min(n, land.size), replace=False)
    X = wrk.shape[2]
    return [(int(i // X), int(i % X)) for i in flat]


def _cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def cpu_baseline(da, wrk, ncells, label, nworkers=None, seed=7):
    from oracle import cpu_farm
    cells = sample_cells(wrk, ncells, seed)
    done, wall, nw = cpu_farm.run_sample(da[0], da[1], wrk, cells, nworkers)
    return {"value": done * NDAYS / wall, "unit": UNIT, "cores": nw, "kind": "port",
            "sample": "%d random land cells of %s x %d days, oracle restatement of step25:126-175 (numpy KED instead of "
                      "rpy2/R gstat), multiprocessing farm, %.1f s" % (done, label, NDAYS, wall),
            "cpu_model": _cpu_model()}, done, wall


_JSON_OUT = None


def _claim_stdout():
    """Rank 0 prints exactly ONE line on stdout.  Libraries write there too (NCCL announces its version on fd 1 when the
    first communicator is created), so fd 1 is pointed at stderr for the rest of the process and the JSON line goes to a
    private duplicate of the original stdout."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def _emit(line):
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()


def _ntiles_arg():
    v = os.environ.get("TWX_BENCH_TILES", str(NTILES_DEFAULT))
    return None if v == "all" else int(v)


def workload_text(ntiles_used, ntiles_all, nland):
    return ("configs[4] (C5): CONUS 30-arcsec grid 3250x7000 with synthetic land mask, %d synthetic stations/var, 365 days "
            "Tmin+Tmax; one step = %d distinct 250x250 tiles (%s of the %d land tiles of Tiler.tile_chks, %d land cells)"
            % (NSTNS_C5, ntiles_used, "all" if ntiles_used == ntiles_all else "a fixed evenly spaced sample",
               ntiles_all, nland))


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path (oracle port; the real one needs
    Python 2 + R/gstat + mpi4py) on all host cores, each step a bounded sample of the same workload."""
    if rank != 0:
        return
    from topowx_b200 import synth
    f, tiler, tiles, nall = c5_tile_list(_ntiles_arg())
    da = c5_stations(f)
    ncells = int(os.environ.get("TWX_REF_CELLS_PER_STEP", "512"))
    done_tot, wall_tot, nw = 0, 0.0, 0
    full = [t for t in tiles]
    for i in range(args.warmup + args.steps):
        t = full[i % len(full)]                                 # a different tile of the list every step
        wrk = synth.make_wrk_chk_grid(f, t[1], t[2], TILE, TILE)
        base, done, wall = cpu_baseline(da, wrk, ncells, "tile %d" % t[0], seed=100 + i)
        nw = base["cores"]
        if i >= args.warmup:
            done_tot += done
            wall_tot += wall
    value = done_tot * NDAYS / wall_tot
    nland = sum(t[3] for t in tiles)
    base = {"value": value, "unit": UNIT, "cores": nw, "kind": "port", "cpu_model": _cpu_model(),
            "sample": "%d steps x %d random land cells of one tile of the list (a different tile per step) x %d days; oracle "
                      "restatement of step25:126-175 (numpy KED instead of rpy2/R gstat), multiprocessing farm"
                      % (args.steps, ncells, NDAYS)}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": wall_tot / args.steps * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "impl": "reference",
            "config": {"workload": workload_text(len(tiles), nall, nland) + "; each reference step = %d-cell sample" % ncells},
            "cpu_baseline": base,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    _emit(line)


class Puller(object):
    """Shared tile counter: the coordinator rank of step25 (step25:293-305) as an atomic counter.  One key per pass."""

    def __init__(self, world):
        self.world = world
        self.local = {}
        self.store = None
        if world > 1:
            import torch.distributed as dist
            self.store = dist.distributed_c10d._get_default_store()

    def next(self, key):
        if self.store is None:
            v = self.local.get(key, 0)
            self.local[key] = v + 1
            return v
        return int(self.store.add("twx_pull_" + key, 1)) - 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--cpu-cells", type=int, default=int(os.environ.get("TWX_CPU_CELLS", "2048")))
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a fixed sample of the last timed step's results to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the CUDA path's results; --impl reference has none")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    _claim_stdout()
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (topowx_b200 has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from topowx_b200 import db, _lib, synth
    from topowx_b200.context import TwxiContext, interp_chunk, interp_chunk_wait
    lib = _lib.lib

    t_setup = time.perf_counter()
    f, tiler, tiles, nall = c5_tile_list(_ntiles_arg())
    NT = len(tiles)
    nland = sum(t[3] for t in tiles)
    da = c5_stations(f)
    ctx = [TwxiContext(d, np.isnan(d.stns[db.BAD]), device=local_rank) for d in da]
    stream = torch.cuda.Stream()
    for c in ctx:
        c.set_stream(stream.cuda_stream)
    # every rank holds every tile of the list (any rank may pull any tile): pinned host copies for the end-to-end leg,
    # device copies for the resident leg
    wrk_h = torch.empty((NT, 32, TILE, TILE), dtype=torch.float64).pin_memory()
    for i, t in enumerate(tiles):
        wrk_h[i] = torch.from_numpy(synth.make_wrk_chk_grid(f, t[1], t[2], TILE, TILE))
    wrk_d = wrk_h.to("cuda")

    def mk(dev):
        kw = dict(device="cuda") if dev else dict(pin_memory=True)
        return dict(tmin=torch.empty((NDAYS, TILE, TILE), dtype=torch.int16, **kw),
                    tmax=torch.empty((NDAYS, TILE, TILE), dtype=torch.int16, **kw),
                    tmin_norm=torch.empty((12, TILE, TILE), dtype=torch.float32, **kw),
                    tmax_norm=torch.empty((12, TILE, TILE), dtype=torch.float32, **kw),
                    tmin_se=torch.empty((12, TILE, TILE), dtype=torch.float32, **kw),
                    tmax_se=torch.empty((12, TILE, TILE), dtype=torch.float32, **kw),
                    ninvalid=torch.empty((TILE, TILE), dtype=torch.int32, **kw),
                    status=torch.empty((TILE, TILE), dtype=torch.uint8, **kw))
    out_d = [mk(True) for _ in range(2)]
    out_h = [mk(False) for _ in range(3)]       # one set of pinned result buffers per chunk in flight (async contract: 3)
    dump = OutputDump(NT) if args.dump_outputs else None
    t_setup = time.perf_counter() - t_setup
    puller = Puller(world)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    pass_id = [0]

    def run_pass(kind, nsteps, dump=None):
        """nsteps passes over the tile list, tiles pulled from the shared counter.  kind 'resident': device buffers, at
        most two tiles in flight per rank; 'e2e': pinned host buffers through twxi_interp_chunk_async (host->device copy of
        the next tile and device->host copy of the previous one overlap the kernels; the library lets two run ahead).
        dump (resident only): takes every tile's results of the last pass."""
        ntile = 0
        with torch.cuda.stream(stream):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            ring = [None, None]
            for step in range(nsteps):
                key = "p%d" % pass_id[0]
                pass_id[0] += 1
                while True:
                    i = puller.next(key)
                    if i >= NT:
                        break
                    if kind == "resident":
                        s = ntile & 1
                        if ring[s] is not None:
                            ring[s].synchronize()               # throttle: a rank never holds more than two tiles
                        interp_chunk(ctx[0], ctx[1], wrk_d[i], out=out_d[s])
                        if dump is not None and step == nsteps - 1:
                            dump.take(i, out_d[s])
                        ev = torch.cuda.Event()
                        ev.record(stream)
                        ring[s] = ev
                    else:
                        interp_chunk(ctx[0], ctx[1], wrk_h[i], out=out_h[ntile % 3], wait=False)
                    ntile += 1
            if kind == "e2e":
                interp_chunk_wait(ctx[0], host_sync=False)       # orders the stream after the last device->host copy
            e1.record(stream)
        e1.synchronize()
        if kind == "e2e":
            interp_chunk_wait(ctx[0], host_sync=True)
        return e0.elapsed_time(e1), ntile

    sampler = ClockSampler(local_rank) if rank == 0 else None
    run_pass("resident", args.warmup)
    barrier()
    if sampler:
        sampler.start()
    lib.twxi_launch_count(1)
    t_wall = time.perf_counter()
    ms_res, nt_res = run_pass("resident", args.steps, dump)
    barrier()
    t_wall = time.perf_counter() - t_wall
    launches = int(lib.twxi_launch_count(0))
    run_pass("e2e", 1)
    barrier()
    ms_e2e, nt_e2e = run_pass("e2e", args.steps)
    barrier()
    clocks = sampler.stop() if sampler else None

    stats = torch.tensor([ms_res, ms_e2e, float(launches), float(nt_res)], dtype=torch.float64, device="cuda")
    if world > 1:
        allst = [torch.zeros_like(stats) for _ in range(world)]
        dist.all_gather(allst, stats)
        allst = torch.stack(allst).cpu().numpy()
    else:
        allst = stats.cpu().numpy()[None, :]
    tot_ms, tot_e2e_ms = float(allst[:, 0].max()), float(allst[:, 1].max())
    launches_all = int(allst[:, 2].sum())
    if dump is not None:
        dump.save(args.dump_outputs, world, rank)

    # ---- per-kernel rooflines: a separate pass with stage events over the first (full-land) tiles of the list ----------
    nroof = min(4, NT)
    flops_ked = flops_gwr = 0.0
    cells_roof = 0
    days_in_month = [int(ctx[0].mth_idx[m].size) for m in range(1, 13)]
    ncand = []
    for i in range(nroof):
        w = wrk_h[i].numpy()
        land = w[2].ravel() != 0
        lat, lon = w[3].ravel()[land], w[4].ravel()[land]
        cells_roof += int(land.sum())
        for c in ctx:
            kn, ka, vario, st = c.nngh_params(lat, lon)
            ok = st == 0
            flops_ked += ked_flops(kn[ok])
            flops_gwr += gwr_flops(ka[ok], days_in_month)
    stage = np.zeros(6)
    lib.twxi_set_stage_timing(1)
    for rep in range(2):
        for i in range(nroof):
            interp_chunk(ctx[0], ctx[1], wrk_d[i], out=out_d[0])
            torch.cuda.synchronize()
            s5 = (C.c_float * 5)()
            lib.twxi_get_stage_ms(s5)
            kk = C.c_float()
            lib.twxi_get_ked_kernel_ms(C.byref(kk))
            if rep:
                stage += np.array(list(s5) + [kk.value])
            if rep:
                cc = C.c_double()
                for c in ctx:
                    lib.twxi_ctx_stat(c.handle, 0, C.byref(cc))
                    ncand.append(cc.value)
    lib.twxi_set_stage_timing(0)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    units = float(nland) * NDAYS
    value = units * args.steps / (tot_ms / 1e3)
    e2e_value = units * args.steps / (tot_e2e_ms / 1e3)
    h2d = NT * 32 * TILE * TILE * 8
    d2h = NT * sum(v.numel() * v.element_size() for v in out_h[0].values())

    dmma, dfma = C.c_double(), C.c_double()
    lib.twxi_measure_fp64_peak(local_rank, C.byref(dmma), C.byref(dfma))
    # independent cross-check of the FP64 peak: cuBLAS DGEMM through torch (library code, not ours), best of 5
    dgemm = None
    try:
        n = 6144
        x = torch.randn(n, n, dtype=torch.float64, device="cuda")
        y = torch.randn(n, n, dtype=torch.float64, device="cuda")
        torch.matmul(x, y)
        best = 1e9
        for _ in range(5):
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            torch.matmul(x, y)
            g1.record()
            g1.synchronize()
            best = min(best, g0.elapsed_time(g1))
        dgemm = 2.0 * n ** 3 / (best / 1e3) / 1e12
        del x, y
    except Exception:
        pass
    ked_ms, krig_ms, gwr_ms, knn_ms = float(stage[5]), float(stage[2]), float(stage[3]), float(stage[0])
    peak = dmma.value
    traffic = _ked_traffic()
    ach = lambda fl, ms: (fl / (ms / 1e3) / 1e12) if ms > 0 else None
    a_ked, a_gwr = ach(flops_ked, ked_ms), ach(flops_gwr, gwr_ms)
    mean_cand = float(np.mean(ncand)) if ncand else None
    flops_knn = 25.0 * (mean_cand or 0.0) * cells_roof * 2
    a_knn = ach(flops_knn, knn_ms)
    peak_note = ("FP64 peak measured in this run by twxi_measure_fp64_peak (DMMA m8n8k4 loop %.1f, DFMA loop %.1f TFLOP/s); "
                 "MEASURED_PEAKS.json has no FP64 entry; nominal B200 FP64 37-40 TFLOP/s" % (dmma.value, dfma.value))
    roofline = {"bound": "tensor", "kernel": "ked_kernel (regression kriging, FP64 DMMA m8n8k4)",
                "achieved": a_ked, "peak": peak, "unit": "TFLOP/s", "frac": (a_ked / peak) if a_ked else None,
                "traffic": traffic["bytes_per_launch_set"] if traffic else None,
                "traffic_source": traffic, "peak_source": peak_note, "fp64_dfma_peak_tflops": dfma.value,
                "fp64_cublas_dgemm_tflops": dgemm,
                "measured_on": "tiles %s of the list (%d land cells), separate pass with CUDA events inside the library"
                               % ([t[0] for t in tiles[:nroof]], cells_roof),
                "algorithmic_flops": flops_ked, "kernel_ms": ked_ms, "stage_ms_incl_gather_sort": krig_ms,
                "launches": "2 variable passes x one launch per size class NB = ceil(n/8) per tile; achieved = sum of their "
                            "algorithmic FLOPs / sum of their CUDA-event durations (twxi_get_ked_kernel_ms)",
                "hbm_floor": {"bytes_per_cell_day": 4, "achieved_gbs": units * 4 * args.steps / (tot_ms / 1e3) / 1e9,
                              "peak_gbs": _measured("hbm_gbs")}}
    rooflines = {
        "ked_kernel": {"bound": "tensor", "achieved": a_ked, "peak": peak, "unit": "TFLOP/s",
                       "frac": (a_ked / peak) if a_ked else None, "ms": ked_ms, "share_of_step": ked_ms / stage[:5].sum()},
        "gwr_kernel": {"bound": "tensor", "achieved": a_gwr, "peak": peak, "unit": "TFLOP/s",
                       "frac": (a_gwr / peak) if a_gwr else None, "ms": gwr_ms, "share_of_step": gwr_ms / stage[:5].sum(),
                       "note": "F_gwr + F_app (SURVEY 8d); latency/gather-bound stage, obs lines from L2",
                       "output_gbs": cells_roof * NDAYS * 2 * 8 / (gwr_ms / 1e3) / 1e9 if gwr_ms > 0 else None},
        "knn_kernels": {"bound": "tensor", "achieved": a_knn, "peak": peak, "unit": "TFLOP/s",
                        "frac": (a_knn / peak) if a_knn else None, "ms": knn_ms, "share_of_step": knn_ms / stage[:5].sum(),
                        "note": "F_knn = 25 flop-equivalents x candidates scanned per cell-variable (SURVEY 8d); mean "
                                "candidates per cell %.0f of %d stations" % (mean_cand or 0, ctx[0].n)},
        "stage_ms": dict(zip(["knn", "nngh_params", "krig", "gwr_daily", "fixer_quantise"],
                             [round(float(x), 3) for x in stage[:5] / nroof])),
    }

    per_rank = {"resident_ms": [round(float(x), 2) for x in allst[:, 0]], "e2e_ms": [round(float(x), 2) for x in allst[:, 1]],
                "tiles_resident": [int(x) for x in allst[:, 3]]}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": tot_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_text(NT, nall, nland), "tiles": NT, "land_cells": nland, "days": NDAYS,
                       "stations_per_var": [int(c.n) for c in ctx],
                       "l2": "not flushed: consecutive tiles are distinct and one tile's working set (6 GB of staged distance "
                             "tiles, 91 MB of output) exceeds the 126 MB L2",
                       "parallelism": "one fixed tile list divided among %d GPU(s) by a shared pull counter, largest tiles "
                                      "first; stations replicated; no collective on the data path" % world,
                       "setup_s": round(t_setup, 1)},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": tot_e2e_ms / args.steps,
                    "mode": "every tile from its own pinned host work chunk into one of three pinned result sets through "
                            "twxi_interp_chunk_async; one timed region per rank from the first submission to the last result "
                            "byte on the host, max over ranks"},
            "gpu_launches": launches_all, "roofline": roofline, "rooflines": rooflines, "clocks": clocks,
            "per_rank": per_rank, "wall_s_timed_region": t_wall}
    if world == 1 and not args.no_secondary:
        line["secondary"] = secondary_runs(ctx, da, tiles, wrk_h, wrk_d, out_d, out_h, stream, lib, args, tiler)
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(da, wrk_h[0].numpy(), args.cpu_cells, "tile %d of the list" % tiles[0][0])[0]
    _emit(line)
    if world > 1:
        dist.destroy_process_group()


def secondary_runs(ctx, da, tiles, wrk_h, wrk_d, out_d, out_h, stream, lib, args, tiler):
    """Figures that are not the headline: C4 (normals only), C3 (leave-one-out at every station), the bytes-on-disk leg,
    and the round-1 workload configs[1] (one interior tile, 2 000 stations) for continuity."""
    import shutil
    import tempfile
    import torch
    from topowx_b200 import db
    from topowx_b200.context import TwxiContext, interp_chunk
    from topowx_b200.interp.tiling import AsyncTileWriter
    sec = {}
    ev = lambda: torch.cuda.Event(enable_timing=True)
    # C4: 12 monthly normals Tmin+Tmax (no daily GWR) on the first 8 tiles of the list
    n4 = min(8, len(tiles))
    o4 = dict(out_d[0], tmin=None, tmax=None)
    with torch.cuda.stream(stream):
        interp_chunk(ctx[0], ctx[1], wrk_d[0], out=o4, daily=False)
        e0, e1 = ev(), ev()
        e0.record(stream)
        for i in range(n4):
            interp_chunk(ctx[0], ctx[1], wrk_d[i], out=o4, daily=False)
        e1.record(stream)
    e1.synchronize()
    ms = e0.elapsed_time(e1)
    cells = sum(t[3] for t in tiles[:n4])
    sec["C4_normals_only"] = {"tiles": n4, "land_cells": cells, "ms": ms, "cell_month_vars_per_s": cells * 24 / (ms / 1e3)}
    # C3: leave-one-out interpolation of the 12 normals at every good station, both variables (step24)
    t0 = time.perf_counter()
    nst = 0
    for c, d in zip(ctx, da):
        s = c.stns
        lst = np.stack([s[db.get_lst_varname(m)] for m in range(1, 13)], axis=1)
        rm = np.arange(c.n, dtype=np.int32).reshape(-1, 1)
        dly, norms, se, var, st = c.interp_points(s[db.LAT], s[db.LON], s[db.ELEV], s[db.TDI], lst, rm_idx=rm, rm_zero=True,
                                                  daily=False)
        nst += int((st == 0).sum())
    dt = time.perf_counter() - t0
    sec["C3_loo_normals"] = {"stations_ok": nst, "wall_s_incl_copies": dt, "station_month_vars_per_s": nst * 12 / dt}
    # ... and with the daily series (what step24 writes per station: daily f8[ndays] + norms[12], step24:67), in batches
    t0 = time.perf_counter()
    nst = 0
    for c in ctx:
        s = c.stns
        lst = np.stack([s[db.get_lst_varname(m)] for m in range(1, 13)], axis=1)
        for i0 in range(0, c.n, 4096):
            sl = slice(i0, min(i0 + 4096, c.n))
            rm = np.arange(sl.start, sl.stop, dtype=np.int32).reshape(-1, 1)
            dly, norms, se, var, st = c.interp_points(s[db.LAT][sl], s[db.LON][sl], s[db.ELEV][sl], s[db.TDI][sl], lst[sl],
                                                      rm_idx=rm, rm_zero=True, daily=True)
            nst += int((st == 0).sum())
    dt = time.perf_counter() - t0
    sec["C3_loo_daily"] = {"stations_ok": nst, "wall_s_incl_copies": dt, "station_days_per_s": nst * NDAYS / dt}
    # bytes on disk: 8 tiles end to end with a background raw writer consuming every result (3 pinned sets in flight)
    tmp = tempfile.mkdtemp(prefix="twx_bench_")
    try:
        from topowx_b200.context import interp_chunk_wait
        days = da[0].days
        aw = AsyncTileWriter(tiler.build_tile_grid_info(), tmp, days, fmt="raw", nthreads=4)
        nd = min(8, len(tiles))
        t0 = time.perf_counter()
        for i in range(nd):
            o = out_h[i % 3]
            interp_chunk(ctx[0], ctx[1], wrk_h[i], out=o, wait=False)
            if i >= 2:                                          # chunk i-2 is complete once chunk i has been submitted
                j = i - 2
                aw.submit(tiler.tile_ids[tiles[j][0]], {k: v.numpy() for k, v in out_h[j % 3].items()}, copy=True)
        interp_chunk_wait(ctx[0], host_sync=True)
        for j in range(max(nd - 2, 0), nd):
            aw.submit(tiler.tile_ids[tiles[j][0]], {k: v.numpy() for k, v in out_h[j % 3].items()}, copy=True)
        nbytes = aw.wait()
        dt = time.perf_counter() - t0
        aw.close()
        cells = sum(t[3] for t in tiles[:nd])
        sec["e2e_to_disk"] = {"tiles": nd, "bytes_on_disk": int(nbytes), "wall_s": dt, "cell_days_per_s": cells * NDAYS / dt,
                              "format": "raw .npy per array (AsyncTileWriter, 4 threads); netCDF needs netCDF4 or scipy"}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    # configs[1]: the round-1 workload
    da1, wrk1 = build_inputs(0)
    ctx1 = [TwxiContext(d, np.isnan(d.stns[db.BAD]), device=torch.cuda.current_device()) for d in da1]
    for c in ctx1:
        c.set_stream(stream.cuda_stream)
    w1 = torch.from_numpy(wrk1).cuda()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    tot = 0.0
    with torch.cuda.stream(stream):
        for i in range(2 + 3):
            flush.fill_(1)
            e0, e1 = ev(), ev()
            e0.record(stream)
            interp_chunk(ctx1[0], ctx1[1], w1, out=out_d[0])
            e1.record(stream)
            e1.synchronize()
            if i >= 2:
                tot += e0.elapsed_time(e1)
    sec["configs1_tile_2000_stations"] = {"ms_per_step": tot / 3, "cell_days_per_s": TILE * TILE * NDAYS / (tot / 3 / 1e3),
                                          "note": "the round-1 headline workload: one interior 250x250 tile, 2000 stations/var, "
                                                  "L2 flushed between steps"}
    for c in ctx1:
        c.close()
    return sec


def _ked_traffic():
    """DRAM bytes of the ked_kernel launches from the committed ncu capture of this round (tools/gpu_traffic.sh)."""
    for name in ("ked_traffic_r02.json", "ked_traffic_r01_k.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                d = json.load(f)
            return {"file": "profiles/" + name, "bytes_per_launch_set": d["dram_bytes_read"] + d["dram_bytes_write"],
                    "commit": d.get("commit"), "workload": d.get("workload", "configs[1] tile, one step")}
        except Exception:
            continue
    return None


def _measured(key):
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f).get(key)
    except Exception:
        return None


if __name__ == "__main__":
    main()

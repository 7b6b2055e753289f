"""Modes of the work-chunk calls that the other GPU tests leave out: the normals-only chunk (daily=False) in every memory
space, the stage-timing slots of the chunk and tile calls, and the launches of a month window.  Run with -m gpu."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

KEYS = ("tmin_norm", "tmax_norm", "tmin_se", "tmax_se", "ninvalid", "status")


@pytest.fixture(scope="module")
def rec():
    """1980-1982 (the 1981-2010 normals start mid-record), a few masked cells."""
    from topowx_b200 import synth, db
    from topowx_b200.context import TwxiContext
    f = synth.Fields()
    days = synth.make_days(1980, 3)
    da = [synth.make_station_db(w, 600, synth.tile_bbox(buf=2.0), f, days, seed=31) for w in (0, 1)]
    ctx = [TwxiContext(d, np.isnan(d.stns[db.BAD])) for d in da]
    wrk = synth.make_wrk_chk(f, synth.TILE_ROW0 + 40, synth.TILE_COL0 + 30, 10, 13)
    wrk[2, 2:4, 5:8] = 0
    return dict(days=days, ctx=ctx, wrk=wrk)


def _np(d):
    return {k: (None if v is None else (v.cpu().numpy() if hasattr(v, "cpu") else np.asarray(v))) for k, v in d.items()}


def test_normals_only_every_memory_space(rec):
    import torch
    from topowx_b200.context import interp_chunk, interp_chunk_wait
    ctx, wrk = rec["ctx"], rec["wrk"]
    host = _np(interp_chunk(ctx[0], ctx[1], wrk, daily=False))
    assert host["tmin"] is None and host["tmax"] is None
    dev = _np(interp_chunk(ctx[0], ctx[1], torch.from_numpy(wrk).cuda(), daily=False))
    assert dev["tmin"] is None and dev["tmax"] is None
    ny, nx = wrk.shape[1:]
    shapes = dict(tmin_norm=((12, ny, nx), torch.float32), tmax_norm=((12, ny, nx), torch.float32),
                  tmin_se=((12, ny, nx), torch.float32), tmax_se=((12, ny, nx), torch.float32),
                  ninvalid=((ny, nx), torch.int32), status=((ny, nx), torch.uint8))
    wrk_pin = torch.from_numpy(wrk).pin_memory()
    outs = [{k: torch.empty(s, dtype=dt).pin_memory() for k, (s, dt) in shapes.items()} for _ in range(3)]
    for o in outs:                                            # three submissions: both staging slots, one reused
        o.update(tmin=None, tmax=None)
        interp_chunk(ctx[0], ctx[1], wrk_pin, out=o, daily=False, wait=False)
    interp_chunk_wait(ctx[0])
    for k in KEYS:
        assert np.array_equal(host[k], dev[k]), k
        for o in outs:
            assert np.array_equal(host[k], o[k].numpy()), k

    daily = _np(interp_chunk(ctx[0], ctx[1], wrk))
    ok_n, ok_d = host["status"] == 0, daily["status"] == 0
    assert ok_n.sum() > 50 and (~ok_n).sum() >= 6
    assert not (ok_d & ~ok_n).any()                           # a cell that fails without dailies fails with them
    both = ok_n & ok_d
    for k in ("tmin_se", "tmax_se"):
        assert np.array_equal(host[k][:, both], daily[k][:, both]), k
    assert (host["ninvalid"][ok_n] == 0).all()
    same = both & (daily["ninvalid"] == 0)                    # no day fixed: the kriged normals stand
    assert same.sum() > 50
    for k in ("tmin_norm", "tmax_norm"):
        assert np.array_equal(host[k][:, same], daily[k][:, same]), k


def _stage_ms(lib):
    s5 = (C.c_float * 5)()
    assert lib.twxi_get_stage_ms(s5) == 0
    return np.array(list(s5), dtype=np.float64)


def test_stage_slots(rec):
    from topowx_b200._lib import lib
    from topowx_b200.context import interp_chunk, tile_begin, tile_days, tile_days_mth, tile_end, MonthGroups
    ctx, wrk, days = rec["ctx"], rec["wrk"], rec["days"]
    lib.twxi_set_stage_timing(1)
    try:
        for daily in (True, False):
            interp_chunk(ctx[0], ctx[1], wrk, daily=daily)
            ms = _stage_ms(lib)
            assert np.isfinite(ms).all() and (ms >= 0).all() and ms.sum() > 0, (daily, ms)
        shape = tile_begin(ctx[0], ctx[1], wrk)
        ms = _stage_ms(lib)
        assert np.isfinite(ms).all() and (ms >= 0).all() and (ms[:3] > 0).all() and ms[4] > 0, ms
        g = MonthGroups(days)
        for n in (45, 300):
            tile_days_mth(ctx[0], ctx[1], n, shape, g)
            ms = _stage_ms(lib)
            assert (ms[:3] == 0).all() and (ms[3:] > 0).all(), ("tile_days_mth", n, ms)
        shape = tile_begin(ctx[0], ctx[1], wrk)
        for n in (45, days.size - 45):
            tile_days(ctx[0], ctx[1], n, shape)
            ms = _stage_ms(lib)
            assert (ms[:3] == 0).all() and (ms[3:] > 0).all(), ("tile_days", n, ms)
        tile_end(ctx[0], ctx[1], shape)
    finally:
        lib.twxi_set_stage_timing(0)


def test_month_window_launches_one_kernel_more(rec):
    from topowx_b200._lib import lib
    from topowx_b200.context import tile_begin, tile_days, tile_days_mth, MonthGroups
    ctx, wrk, days = rec["ctx"], rec["wrk"], rec["days"]
    counts = {}
    for what in ("days", "mth"):
        shape = tile_begin(ctx[0], ctx[1], wrk)
        g = MonthGroups(days)
        for n in (45, 1, 400):
            lib.twxi_launch_count(1)
            if what == "days":
                tile_days(ctx[0], ctx[1], n, shape)
            else:
                tile_days_mth(ctx[0], ctx[1], n, shape, g)
            counts[what, n] = int(lib.twxi_launch_count(0))
    for n in (45, 1, 400):
        assert counts["days", n] > 0
        assert counts["mth", n] == counts["days", n] + 1, (n, counts)

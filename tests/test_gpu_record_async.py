"""Asynchronous day windows (twxi_tile_begin_async / _days[_mth]_async / _end_async): the bytes of the synchronous calls
for every partition, the ownership rule (a submission's buffers are complete once two further submissions have been made,
chunks and tile calls counted together), tiles back to back, interleaved calls, misuse and device buffers.  Run with
-m gpu."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

KEYS = ("tmin_norm", "tmax_norm", "tmin_se", "tmax_se", "ninvalid", "status")
ERR_ARG, ERR_STATE = -1, -3
SENTINEL = 0x5A                                                       # byte pattern of a buffer not yet written


@pytest.fixture(scope="module")
def rec():
    """1979-1983 (1 826 days: leap year 1980, the 1981-2010 groups start mid-record) with the fixer heavily active and
    masked cells, plus a second chunk for the back-to-back and interleaving cases."""
    import torch
    from topowx_b200 import synth, db
    from topowx_b200.context import TwxiContext, interp_chunk
    f = synth.Fields(dtr_override=0.3)
    days = synth.make_days(1979, 5)
    da = [synth.make_station_db(w, 700, synth.tile_bbox(buf=2.0), f, days, seed=77) for w in (0, 1)]
    ctx = [TwxiContext(d, np.isnan(d.stns[db.BAD])) for d in da]
    wrk = synth.make_wrk_chk(f, synth.TILE_ROW0 + 10, synth.TILE_COL0 + 20, 12, 15)
    wrk[2, 3:5, 4:7] = 0                                              # masked cells
    ref = interp_chunk(ctx[0], ctx[1], wrk)
    assert (ref["status"] == 255).sum() == 6 and ref["ninvalid"][ref["status"] == 0].min() > 0
    other = synth.make_wrk_chk(f, synth.TILE_ROW0 + 100, synth.TILE_COL0 + 60, 5, 7)
    other_ref = interp_chunk(ctx[0], ctx[1], other)
    return dict(days=days, da=da, ctx=ctx, wrk=wrk, ref=ref, other=other, other_ref=other_ref,
                wrk_p=torch.from_numpy(wrk).pin_memory(), other_p=torch.from_numpy(other).pin_memory())


def poison(t):
    import torch
    t.view(torch.uint8).fill_(SENTINEL)
    return t


def pinned(shape, dt):
    import torch
    return poison(torch.empty(shape, dtype=getattr(torch, dt)).pin_memory())


def mth_out(groups, n, shape):
    g0, g1 = groups.completed(n)
    return dict(day_out(n, shape), tmin_mth=pinned((g1 - g0,) + shape, "float32"),
                tmax_mth=pinned((g1 - g0,) + shape, "float32"))


def day_out(n, shape):
    return dict(tmin=pinned((n,) + shape, "int16"), tmax=pinned((n,) + shape, "int16"))


def fin_out(shape):
    return dict(tmin_norm=pinned((12,) + shape, "float32"), tmax_norm=pinned((12,) + shape, "float32"),
                tmin_se=pinned((12,) + shape, "float32"), tmax_se=pinned((12,) + shape, "float32"),
                ninvalid=pinned(shape, "int32"), status=pinned(shape, "uint8"))


def host(d):
    return {k: (v.cpu().numpy() if hasattr(v, "cpu") else np.asarray(v)) for k, v in d.items() if k != "mth_groups"}


def same(ref, got, keys, what):
    for k in keys:
        assert np.array_equal(np.asarray(ref[k]), np.asarray(got[k])), (what, k)


def wait(ctx):
    from topowx_b200.context import interp_chunk_wait
    interp_chunk_wait(ctx[0])


def year_sizes(days):
    return np.unique(days["YEAR"], return_counts=True)[1].tolist()


def run_async(ctx, wrk_p, sizes, shape):
    """begin, every window and end submitted without waiting, each into its own pinned set; then the wait."""
    from topowx_b200.context import tile_begin, tile_days, tile_end
    tile_begin(ctx[0], ctx[1], wrk_p, wait=False)
    parts = [tile_days(ctx[0], ctx[1], n, shape, out=day_out(n, shape), wait=False) for n in sizes]
    fin = tile_end(ctx[0], ctx[1], shape, out=fin_out(shape), wait=False)
    wait(ctx)
    out = host(fin)
    for k in ("tmin", "tmax"):
        out[k] = np.concatenate([p[k].numpy() for p in parts])
    return out


def test_partitions_are_byte_identical(rec):
    days, ref, ctx = rec["days"], rec["ref"], rec["ctx"]
    nd = days.size
    d1981 = int(np.searchsorted(days["YEAR"], 1981))
    in_month = d1981 + 59 + 10                                        # 1981-03-11
    parts = {
        "one window": [nd],
        "1-day windows, then the rest": [1] * 40 + [nd - 40],
        "97-day windows": [97] * (nd // 97) + [nd % 97],
        "split inside a month": [in_month, nd - in_month],
        "split at 1981-01-01": [d1981, nd - d1981],
    }
    for what, sizes in parts.items():
        out = run_async(ctx, rec["wrk_p"], sizes, (12, 15))
        same(ref, out, ("tmin", "tmax") + KEYS, what)


def test_month_windows_equal_the_synchronous_call(rec):
    from topowx_b200.context import tile_begin, tile_days_mth, tile_end, MonthGroups
    days, ctx, shape = rec["days"], rec["ctx"], (12, 15)
    nd = days.size
    for sizes in (year_sizes(days), [97] * (nd // 97) + [nd % 97]):
        tile_begin(ctx[0], ctx[1], rec["wrk"])
        g = MonthGroups(days)
        sync = [host(tile_days_mth(ctx[0], ctx[1], n, shape, g)) for n in sizes]
        sync_fin = host(tile_end(ctx[0], ctx[1], shape))
        tile_begin(ctx[0], ctx[1], rec["wrk_p"], wait=False)
        g = MonthGroups(days)
        parts = []
        for n in sizes:
            g0, g1 = g.completed(n)
            parts.append(tile_days_mth(ctx[0], ctx[1], n, shape, g, out=mth_out(g, n, shape), wait=False))
            assert len(parts[-1]["mth_groups"]) == g1 - g0                     # nmth is known at submission
        fin = tile_end(ctx[0], ctx[1], shape, out=fin_out(shape), wait=False)
        wait(ctx)
        for s, p in zip(sync, parts):
            same(s, host(p), ("tmin", "tmax", "tmin_mth", "tmax_mth"), "months")
        same(sync_fin, host(fin), KEYS, "months end")
        same(rec["ref"], dict(tmin=np.concatenate([s["tmin"] for s in sync])), ("tmin",), "months dailies")


def test_three_sets_carry_the_stream(rec):
    """Window t's set is read right after window t+2 is submitted, with no wait; the sets are then reused."""
    from topowx_b200.context import tile_begin, tile_days, tile_end
    ctx, ref, nd, shape = rec["ctx"], rec["ref"], rec["days"].size, (12, 15)
    sizes = [97] * (nd // 97) + [nd % 97]
    sets = [day_out(97, shape) for _ in range(3)]
    tile_begin(ctx[0], ctx[1], rec["wrk_p"], wait=False)
    subs, d0 = [], 0                                                  # (set, first day, days) per window
    for t, n in enumerate(sizes):
        st = sets[t % 3]
        for v in st.values():                                         # window t-3, checked already, leaves no trace
            poison(v)
        out = {k: v[:n] for k, v in st.items()}
        tile_days(ctx[0], ctx[1], n, shape, out=out, wait=False)
        subs.append((out, d0, n))
        d0 += n
        if t >= 2:                                                    # window t-2 is complete now
            o, a, m = subs[t - 2]
            for k in ("tmin", "tmax"):
                assert np.array_equal(o[k].numpy(), np.asarray(ref[k])[a:a + m]), ("after t+2", t - 2, k)
    fin = tile_end(ctx[0], ctx[1], shape, out=fin_out(shape), wait=False)
    wait(ctx)
    for o, a, m in subs[-2:]:
        for k in ("tmin", "tmax"):
            assert np.array_equal(o[k].numpy(), np.asarray(ref[k])[a:a + m]), ("after the wait", a, k)
    same(ref, host(fin), KEYS, "end")


def test_tiles_back_to_back_and_a_chunk_between(rec):
    """Tile B's begin follows tile A's end at once; a chunk submitted between two tiles and a kriging call between two
    windows change no byte, and the t+2 rule counts chunks and tile calls together."""
    from topowx_b200.context import tile_begin, tile_days, tile_end, interp_chunk
    ctx, days = rec["ctx"], rec["days"]
    ys = year_sizes(days)
    sa, sb = (12, 15), (5, 7)
    tile_begin(ctx[0], ctx[1], rec["wrk_p"], wait=False)
    pa = []
    for i, n in enumerate(ys):
        pa.append(tile_days(ctx[0], ctx[1], n, sa, out=day_out(n, sa), wait=False))
        if i == 1:                                                    # a synchronous call on the pair between windows
            ctx[0].krig(np.array([40.0]), np.array([-105.0]), np.array([1600.0]), np.full(12, 10.0))
    fa = tile_end(ctx[0], ctx[1], sa, out=fin_out(sa), wait=False)
    # a chunk on the same slots: end A = t, chunk = t+1, begin B = t+2
    ch = dict(tmin=pinned((days.size,) + sb, "int16"), tmax=pinned((days.size,) + sb, "int16"), **fin_out(sb))
    interp_chunk(ctx[0], ctx[1], rec["other_p"], out=ch, wait=False)
    tile_begin(ctx[0], ctx[1], rec["other_p"], wait=False)
    same(rec["ref"], host(fa), KEYS, "end of A after two further submissions")
    pb = [tile_days(ctx[0], ctx[1], n, sb, out=day_out(n, sb), wait=False) for n in ys]
    same(rec["other_ref"], host(ch), ("tmin", "tmax") + KEYS, "chunk after two further submissions")
    fb = tile_end(ctx[0], ctx[1], sb, out=fin_out(sb), wait=False)
    wait(ctx)
    for p, ref, fin in ((pa, rec["ref"], fa), (pb, rec["other_ref"], fb)):
        got = dict(host(fin), tmin=np.concatenate([x["tmin"].numpy() for x in p]),
                   tmax=np.concatenate([x["tmax"].numpy() for x in p]))
        same(ref, got, ("tmin", "tmax") + KEYS, "back to back")


def test_misuse_gives_the_synchronous_errors(rec):
    from topowx_b200 import _lib
    from topowx_b200.context import tile_begin, tile_days, tile_days_mth, tile_end, MonthGroups
    ctx, ref, days, shape = rec["ctx"], rec["ref"], rec["days"], (12, 15)
    nd = days.size
    lib = _lib.lib
    h0, h1 = ctx[0].handle, ctx[1].handle

    def both(code, call_async, call_sync):
        """The async call and its synchronous twin, in the same state, fail with the same code and message."""
        msgs = []
        for fn in (call_async, call_sync):
            with pytest.raises(_lib.TwxiError, match="libtwxi error %d:" % code) as e:
                fn()
            msgs.append(str(e.value))
        assert msgs[0] == msgs[1]

    def days_raw(fn, n, o):
        return lambda: _lib.check(fn(h0, h1, n, _lib.ptr(o["tmin"][:n]), _lib.ptr(o["tmax"][:n]), _lib.MEM_HOST))

    big = day_out(nd, shape)
    # no open tile: the last one was ended
    run_async(ctx, rec["wrk_p"], [nd], shape)
    both(ERR_STATE, days_raw(lib.twxi_tile_days_async, 5, big), days_raw(lib.twxi_tile_days, 5, big))
    fo = fin_out(shape)
    end_raw = lambda fn: lambda: _lib.check(fn(h0, h1, *[_lib.ptr(fo[k]) for k in KEYS], _lib.MEM_HOST))
    both(ERR_STATE, end_raw(lib.twxi_tile_end_async), end_raw(lib.twxi_tile_end))

    nm = C.c_int32(-1)
    mo = dict(tmin_mth=pinned((12,) + shape, "float32"), tmax_mth=pinned((12,) + shape, "float32"))

    def mth_raw(fn, max_mth):
        return lambda: _lib.check(fn(h0, h1, 100, _lib.ptr(big["tmin"][:100]), _lib.ptr(big["tmax"][:100]), max_mth,
                                     _lib.ptr(mo["tmin_mth"]), _lib.ptr(mo["tmax_mth"]), C.byref(nm), _lib.MEM_HOST))

    # more days than remain, max_mth too small; each failure leaves the tile as it was and counts as no submission
    tile_begin(ctx[0], ctx[1], rec["wrk_p"], wait=False)                                # t
    g = MonthGroups(days)
    a = tile_days_mth(ctx[0], ctx[1], 400, shape, g, out=mth_out(g, 400, shape), wait=False)   # t+1
    both(ERR_ARG, days_raw(lib.twxi_tile_days_async, nd - 399, big), days_raw(lib.twxi_tile_days, nd - 399, big))
    g0, g1 = g.completed(100)
    assert g1 - g0 >= 2
    both(ERR_ARG, mth_raw(lib.twxi_tile_days_mth_async, g1 - g0 - 1), mth_raw(lib.twxi_tile_days_mth, g1 - g0 - 1))
    b = tile_days_mth(ctx[0], ctx[1], 500, shape, g, out=mth_out(g, 500, shape), wait=False)   # t+2
    c = tile_days_mth(ctx[0], ctx[1], nd - 900, shape, g, out=mth_out(g, nd - 900, shape), wait=False)   # t+3
    for k in ("tmin", "tmax"):                                        # window t+1 after two successful submissions
        assert np.array_equal(a[k].numpy(), np.asarray(ref[k])[:400]), k
    fin = tile_end(ctx[0], ctx[1], shape, out=fin_out(shape), wait=False)
    for k in ("tmin", "tmax"):
        assert np.array_equal(b[k].numpy(), np.asarray(ref[k])[400:900]), k
    wait(ctx)
    for k in ("tmin", "tmax"):
        assert np.array_equal(c[k].numpy(), np.asarray(ref[k])[900:]), k
    same(ref, host(fin), KEYS, "after the errors")

    # _mth after a plain window of the same tile, then the observation record replaced after begin
    tile_begin(ctx[0], ctx[1], rec["wrk_p"], wait=False)
    tile_days(ctx[0], ctx[1], 10, shape, out=day_out(10, shape), wait=False)
    both(ERR_STATE, mth_raw(lib.twxi_tile_days_mth_async, 12), mth_raw(lib.twxi_tile_days_mth, 12))
    ctx[0].set_obs(rec["da"][0])
    both(ERR_STATE, days_raw(lib.twxi_tile_days_async, 10, big), days_raw(lib.twxi_tile_days, 10, big))
    both(ERR_STATE, end_raw(lib.twxi_tile_end_async), end_raw(lib.twxi_tile_end))
    out = run_async(ctx, rec["wrk_p"], year_sizes(days), shape)      # a valid stream right after
    same(ref, out, ("tmin", "tmax") + KEYS, "after set_obs")


def test_device_buffers(rec):
    import torch
    from topowx_b200.context import tile_begin, tile_days, tile_end
    ctx, days, shape = rec["ctx"], rec["days"], (12, 15)
    w = torch.from_numpy(rec["wrk"]).cuda()
    dev = w.device
    got = {}
    for wt in (True, False):
        tile_begin(ctx[0], ctx[1], w, wait=wt)
        parts = [tile_days(ctx[0], ctx[1], n, shape, device=dev, wait=wt) for n in year_sizes(days)]
        fin = tile_end(ctx[0], ctx[1], shape, device=dev, wait=wt)
        torch.cuda.synchronize()
        got[wt] = dict(host(fin), tmin=np.concatenate([p["tmin"].cpu().numpy() for p in parts]),
                       tmax=np.concatenate([p["tmax"].cpu().numpy() for p in parts]))
    same(got[True], got[False], ("tmin", "tmax") + KEYS, "device buffers")
    same(rec["ref"], got[False], ("tmin", "tmax") + KEYS, "device buffers vs whole record")

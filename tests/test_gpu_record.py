"""Multi-year records in day windows (twxi_tile_begin / _days / _end): every partition of the record gives the bytes of
twxi_interp_chunk, the record is right against the oracle over five years, and misuse is reported.  Run with -m gpu."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import twx_oracle as o          # noqa: E402  (checker only)

TOL_C = 1e-4
KEYS = ("tmin_norm", "tmax_norm", "tmin_se", "tmax_se", "ninvalid", "status")


@pytest.fixture(scope="module")
def rec():
    """1979-1983 (1 826 days: leap year 1980, the 1981-2010 groups start mid-record) with the fixer heavily active."""
    from topowx_b200 import synth, db
    from topowx_b200.context import TwxiContext, interp_chunk
    f = synth.Fields(dtr_override=0.3)
    days = synth.make_days(1979, 5)
    da = [synth.make_station_db(w, 700, synth.tile_bbox(buf=2.0), f, days, seed=77) for w in (0, 1)]
    ctx = [TwxiContext(d, np.isnan(d.stns[db.BAD])) for d in da]
    wrk = synth.make_wrk_chk(f, synth.TILE_ROW0 + 10, synth.TILE_COL0 + 20, 12, 15)
    wrk[2, 3:5, 4:7] = 0                                              # masked cells
    ref = interp_chunk(ctx[0], ctx[1], wrk)
    return dict(f=f, days=days, da=da, ctx=ctx, wrk=wrk, ref=ref, synth=synth, db=db)


def _windows(ctx, wrk, sizes, device=False):
    import torch
    from topowx_b200.context import tile_begin, tile_days, tile_end
    w = torch.from_numpy(wrk).cuda() if device else wrk
    shape = tile_begin(ctx[0], ctx[1], w)
    parts = [tile_days(ctx[0], ctx[1], n, shape, device=w.device if device else None) for n in sizes]
    fin = tile_end(ctx[0], ctx[1], shape, device=w.device if device else None)
    host = (lambda a: a.cpu().numpy()) if device else np.asarray
    out = {k: host(v) for k, v in fin.items()}
    for k in ("tmin", "tmax"):
        out[k] = np.concatenate([host(p[k]) for p in parts])
    return out, [{k: host(p[k]) for k in ("tmin", "tmax")} for p in parts]


def _assert_identical(ref, out, what):
    for k in ("tmin", "tmax") + KEYS:
        assert np.array_equal(np.asarray(ref[k]), out[k]), (what, k)


def _year_sizes(days):
    return np.unique(days["YEAR"], return_counts=True)[1].tolist()


def test_partitions_are_byte_identical(rec):
    days, ref = rec["days"], rec["ref"]
    nd = days.size
    assert nd == 1826
    assert (ref["status"] == 255).sum() == 6 and (ref["status"] == 0).sum() > 150
    assert ref["ninvalid"][ref["status"] == 0].min() > 0                      # the fixer really ran
    d1981 = int(np.searchsorted(days["YEAR"], 1981))
    in_month = d1981 + 59 + 10                                                # 1981-03-11
    parts = {
        "one window": [nd],
        "1-day windows, then the rest": [1] * 40 + [nd - 40],
        "97-day windows": [97] * (nd // 97) + [nd % 97],
        "split inside a month": [in_month, nd - in_month],
        "split at 1981-01-01": [d1981, nd - d1981],
    }
    for what, sizes in parts.items():
        assert sum(sizes) == nd
        out, _ = _windows(rec["ctx"], rec["wrk"], sizes)
        _assert_identical(ref, out, what)
    out, _ = _windows(rec["ctx"], rec["wrk"], _year_sizes(days), device=True)  # calendar years, device buffers
    _assert_identical(ref, out, "calendar years")


def test_stream_years_and_oracle_over_five_years(rec):
    """PtInterpTair.interp_chunk_stream by calendar year against the oracle on a few cells of the five-year record: the
    first GPU-vs-oracle check over more than one year (leap day, normals recomputed over 1981-1983)."""
    from topowx_b200.interp import PtInterpTair
    da, wrk, days = rec["da"], rec["wrk"], rec["days"]
    pti = PtInterpTair(da[0], da[1])
    s = pti.interp_chunk_stream(wrk)
    tmin, tmax, day0s = [], [], []
    for d0, out in s.years():
        day0s.append(d0)
        tmin.append(out["tmin"])
        tmax.append(out["tmax"])
    fin = s.finish()
    assert day0s == np.concatenate([[0], np.cumsum(_year_sizes(days))[:-1]]).tolist()
    got = dict(fin, tmin=np.concatenate(tmin), tmax=np.concatenate(tmax))
    _assert_identical(rec["ref"], got, "interp_chunk_stream")
    cells = [(0, 0), (6, 9), (11, 14)]
    opti = o.PtInterpTair(*[o.StationDb(d.stns, d.var, d.days) for d in da])
    ref = o.interp_chunk(opti, wrk, cells=cells)
    for (r, c) in cells:
        assert ref["status"][r, c] == got["status"][r, c] == 0
        assert ref["ninvalid"][r, c] > 5 and ref["ninvalid"][r, c] == got["ninvalid"][r, c]
        for k in ("tmin", "tmax"):
            assert np.abs(got[k][:, r, c].astype(int) - ref[k][:, r, c].astype(int)).max() <= 1, (r, c, k)
        for k in ("tmin_norm", "tmax_norm", "tmin_se", "tmax_se"):
            assert np.abs(got[k][:, r, c] - ref[k][:, r, c]).max() < TOL_C, (r, c, k)


def test_fixer_failure_is_decided_in_a_one_day_first_window():
    """'No valid tmin/tmax in window' (dtr forced to -1.2 C) on a two-year record: a first window of one day, then years.
    Status, ninvalid and every window equal the whole-record call; failed cells are fill in every window."""
    from topowx_b200 import synth, db
    from topowx_b200.context import TwxiContext, interp_chunk
    f = synth.Fields(dtr_override=-1.2)
    days = synth.make_days(1995, 2)
    da = [synth.make_station_db(w, 700, synth.tile_bbox(buf=2.0), f, days, seed=78) for w in (0, 1)]
    ctx = [TwxiContext(d, np.isnan(d.stns[db.BAD])) for d in da]
    wrk = synth.make_wrk_chk(f, synth.TILE_ROW0 + 30, synth.TILE_COL0 + 40, 2, 3)
    ref = interp_chunk(ctx[0], ctx[1], wrk)
    bad = ref["status"] == o.ST_FIXER_EMPTY
    assert bad.any()
    ys = _year_sizes(days)                                            # 365, 366
    sizes = [1, ys[0] - 1] + ys[1:]
    out, parts = _windows(ctx, wrk, sizes)
    _assert_identical(ref, out, "1 + years")
    for p in parts:
        assert np.all(p["tmin"][:, bad] == -32767) and np.all(p["tmax"][:, bad] == -32767)
    assert np.all(out["ninvalid"][bad] == -2147483647)


def test_interleaved_calls_and_misuse(rec):
    from topowx_b200 import _lib
    from topowx_b200.context import TwxiContext, interp_chunk, tile_begin, tile_days, tile_end
    ctx, wrk, ref, nd = rec["ctx"], rec["wrk"], rec["ref"], rec["days"].size
    synth, db = rec["synth"], rec["db"]
    other = synth.make_wrk_chk(rec["f"], synth.TILE_ROW0 + 100, synth.TILE_COL0 + 60, 5, 7)
    other_ref = interp_chunk(ctx[0], ctx[1], other)
    # another chunk on the same contexts between two windows: the stream's output is unchanged
    shape = tile_begin(ctx[0], ctx[1], wrk)
    a = tile_days(ctx[0], ctx[1], 400, shape)
    mid = interp_chunk(ctx[0], ctx[1], other)
    b = tile_days(ctx[0], ctx[1], nd - 400, shape)
    fin = tile_end(ctx[0], ctx[1], shape)
    _assert_identical(ref, dict(fin, tmin=np.concatenate([a["tmin"], b["tmin"]]),
                                tmax=np.concatenate([a["tmax"], b["tmax"]])), "interleaved")
    _assert_identical(other_ref, {k: np.asarray(v) for k, v in mid.items()}, "the call in between")

    def err(code):
        return pytest.raises(_lib.TwxiError, match="libtwxi error %d:" % code)
    ERR_ARG, ERR_STATE = -1, -3
    with err(ERR_STATE):                                  # no open tile: the last one was ended
        tile_days(ctx[0], ctx[1], 1, shape)
    with err(ERR_STATE):
        tile_end(ctx[0], ctx[1], shape)
    shape = tile_begin(ctx[0], ctx[1], wrk)
    with err(ERR_STATE):                                  # end before every day was emitted
        tile_end(ctx[0], ctx[1], shape)
    tile_days(ctx[0], ctx[1], nd - 5, shape)
    with err(ERR_ARG):                                    # more days than remain
        tile_days(ctx[0], ctx[1], 6, shape)
    with err(ERR_ARG):
        tile_days(ctx[0], ctx[1], 0, shape)
    third = TwxiContext(rec["da"][1], np.isnan(rec["da"][1].stns[db.BAD]))
    with err(ERR_ARG):                                    # another ctx_tmax than at begin
        tile_days(ctx[0], third, 5, shape)
    with err(ERR_ARG):
        tile_end(ctx[0], third, shape)
    last = tile_days(ctx[0], ctx[1], 5, shape)            # the failed calls changed nothing
    assert np.array_equal(last["tmin"], np.asarray(ref["tmin"])[nd - 5:])
    tile_end(ctx[0], ctx[1], shape)
    # a new begin discards an open tile
    shape = tile_begin(ctx[0], ctx[1], other)
    tile_days(ctx[0], ctx[1], 10, shape)
    out, _ = _windows(ctx, wrk, [nd])
    _assert_identical(ref, out, "after a discarded tile")
    # the observation record replaced after begin
    shape = tile_begin(ctx[0], ctx[1], wrk)
    tile_days(ctx[0], ctx[1], 10, shape)
    ctx[1].set_obs(rec["da"][1])
    with err(ERR_STATE):
        tile_days(ctx[0], ctx[1], 10, shape)
    with err(ERR_STATE):
        tile_end(ctx[0], ctx[1], shape)

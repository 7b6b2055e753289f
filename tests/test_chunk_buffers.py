"""Argument checks of the chunk and tile wrappers in context.py (CPU only).

The contexts are stubs with ``handle = None``: a call that passes every Python check reaches the C entry point with a NULL
context, which returns TWXI_ERR_ARG before it touches CUDA, so it raises TwxiError instead of ValueError."""
import types

import numpy as np
import pytest

NY, NX, ND = 3, 4, 40


@pytest.fixture(scope="module")
def cx():
    from topowx_b200 import build
    build.build_lib()
    from topowx_b200 import context
    return context


@pytest.fixture(scope="module")
def TwxiError(cx):
    from topowx_b200._lib import TwxiError
    return TwxiError


def ctx(ndays=ND):
    return types.SimpleNamespace(ndays=ndays, handle=None)


def fake_device(a):
    """Shape and dtype of ``a`` in device memory, as context.py sees a CUDA tensor."""
    return types.SimpleNamespace(shape=a.shape, dtype=a.dtype, is_cuda=True, device="cuda:0")


def wrk(dtype=np.float64, planes=32):
    return np.zeros((planes, NY, NX), dtype=dtype)


def chunk_out(nd=ND, daily=True):
    o = dict(tmin_norm=np.empty((12, NY, NX), np.float32), tmax_norm=np.empty((12, NY, NX), np.float32),
             tmin_se=np.empty((12, NY, NX), np.float32), tmax_se=np.empty((12, NY, NX), np.float32),
             ninvalid=np.empty((NY, NX), np.int32), status=np.empty((NY, NX), np.uint8))
    o["tmin"] = np.empty((nd, NY, NX), np.int16) if daily else None
    o["tmax"] = np.empty((nd, NY, NX), np.int16) if daily else None
    return o


# ---- interp_chunk --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("w", [wrk(planes=31), np.zeros((32, NY * NX)), wrk(np.float32)], ids=["planes", "2d", "f4"])
def test_interp_chunk_rejects_wrk_chk(cx, w):
    with pytest.raises(ValueError, match="wrk_chk must be"):
        cx.interp_chunk(ctx(), ctx(), w)


def test_interp_chunk_record_lengths(cx, TwxiError):
    with pytest.raises(ValueError, match="different length"):
        cx.interp_chunk(ctx(ND), ctx(ND + 1), wrk())
    with pytest.raises(TwxiError):                            # normals only: the records may differ
        cx.interp_chunk(ctx(ND), ctx(ND + 1), wrk(), daily=False)


@pytest.mark.parametrize("key", ["tmin", "tmax", "tmin_norm", "tmax_se", "ninvalid", "status"])
def test_interp_chunk_missing_buffer(cx, key):
    out = chunk_out()
    out[key] = None
    with pytest.raises(ValueError, match="is missing"):
        cx.interp_chunk(ctx(), ctx(), wrk(), out=out)
    del out[key]
    with pytest.raises(ValueError, match="is missing"):
        cx.interp_chunk(ctx(), ctx(), wrk(), out=out)


@pytest.mark.parametrize("key,bad", [("tmin", np.empty((ND, NY, NX), np.int32)),
                                     ("tmax", np.empty((ND - 1, NY, NX), np.int16)),
                                     ("tmin_norm", np.empty((12, NY, NX), np.float64)),
                                     ("tmax_se", np.empty((12, NX, NY), np.float32)),
                                     ("ninvalid", np.empty((NY, NX), np.int64)),
                                     ("status", np.empty((NY * NX,), np.uint8))])
def test_interp_chunk_bad_buffer(cx, key, bad):
    out = chunk_out()
    out[key] = bad
    with pytest.raises(ValueError, match="must be"):
        cx.interp_chunk(ctx(), ctx(), wrk(), out=out)
    out = chunk_out(daily=False)                              # a given tmin / tmax is checked without daily too
    if key in ("tmin", "tmax"):
        out[key] = bad
        with pytest.raises(ValueError, match="must be"):
            cx.interp_chunk(ctx(), ctx(), wrk(), out=out, daily=False)


@pytest.mark.parametrize("key", ["tmin", "tmin_norm", "status"])
def test_interp_chunk_memory_space(cx, key):
    out = chunk_out()
    out[key] = fake_device(out[key])
    with pytest.raises(ValueError, match="same memory space as wrk_chk"):
        cx.interp_chunk(ctx(), ctx(), wrk(), out=out)
    out = chunk_out()                                         # all buffers on the host, the chunk on the device
    with pytest.raises(ValueError, match="same memory space as wrk_chk"):
        cx.interp_chunk(ctx(), ctx(), fake_device(wrk()), out=out)


@pytest.mark.parametrize("wait", [True, False])
def test_interp_chunk_valid_reaches_the_library(cx, TwxiError, wait):
    for kw in (dict(), dict(out=chunk_out()), dict(daily=False), dict(daily=False, out=chunk_out(daily=False))):
        with pytest.raises(TwxiError):
            cx.interp_chunk(ctx(), ctx(), wrk(), wait=wait, **kw)


def test_interp_chunk_one_of_tmin_tmax_without_daily(cx, TwxiError):
    out = chunk_out()
    out["tmax"] = None                                        # checked by the library: both or neither
    with pytest.raises(TwxiError):
        cx.interp_chunk(ctx(), ctx(), wrk(), out=out, daily=False)


@pytest.mark.parametrize("daily", [True, False])
def test_interp_chunk_default_buffers(cx, monkeypatch, daily):
    calls = []

    class Lib(object):
        def __getattr__(self, name):
            return lambda *a: calls.append((name, a)) or 0
    monkeypatch.setattr(cx, "lib", Lib())
    out = cx.interp_chunk(ctx(), ctx(), wrk(), daily=daily)
    assert calls[0][0] == "twxi_interp_chunk"
    want = dict(tmin=("int16", (ND, NY, NX)), tmax=("int16", (ND, NY, NX)), tmin_norm=("float32", (12, NY, NX)),
                tmax_norm=("float32", (12, NY, NX)), tmin_se=("float32", (12, NY, NX)),
                tmax_se=("float32", (12, NY, NX)), ninvalid=("int32", (NY, NX)), status=("uint8", (NY, NX)))
    assert list(out) == list(want)
    for k, (dt, shp) in want.items():
        if not daily and k in ("tmin", "tmax"):
            assert out[k] is None
            continue
        assert isinstance(out[k], np.ndarray) and out[k].dtype == dt and out[k].shape == shp, k


# ---- tile windows and end ------------------------------------------------------------------------------------------
def days_out(nd, nm=None):
    o = dict(tmin=np.empty((nd, NY, NX), np.int16), tmax=np.empty((nd, NY, NX), np.int16))
    if nm is not None:
        o.update(tmin_mth=np.empty((nm, NY, NX), np.float32), tmax_mth=np.empty((nm, NY, NX), np.float32))
    return o


def end_out():
    o = chunk_out()
    del o["tmin"], o["tmax"]
    return o


def groups():
    from topowx_b200 import synth
    from topowx_b200.context import MonthGroups
    return MonthGroups(synth.make_days(1995, 1))


def test_tile_begin_checks(cx, TwxiError):
    with pytest.raises(ValueError, match="wrk_chk must be"):
        cx.tile_begin(ctx(), ctx(), wrk(np.float32))
    with pytest.raises(ValueError, match="different length"):
        cx.tile_begin(ctx(ND), ctx(ND + 1), wrk())
    with pytest.raises(TwxiError):
        cx.tile_begin(ctx(), ctx(), wrk())


def test_tile_days_checks(cx, TwxiError):
    for key, bad in (("tmin", np.empty((7, NY, NX), np.int32)), ("tmax", np.empty((6, NY, NX), np.int16)),
                     ("tmin", None)):
        out = days_out(7)
        out[key] = bad
        with pytest.raises(ValueError):
            cx.tile_days(ctx(), ctx(), 7, (NY, NX), out=out)
    out = days_out(7)
    out["tmax"] = fake_device(out["tmax"])
    with pytest.raises(ValueError, match="same memory space as the other result buffers"):
        cx.tile_days(ctx(), ctx(), 7, (NY, NX), out=out)
    for kw in (dict(), dict(out=days_out(7))):
        with pytest.raises(TwxiError):
            cx.tile_days(ctx(), ctx(), 7, (NY, NX), **kw)


def test_tile_days_mth_checks(cx, TwxiError):
    g = groups()
    nd = 45                                                   # completes January
    assert g.completed(nd) == (0, 1)
    for key, bad in (("tmin_mth", np.empty((2, NY, NX), np.float32)), ("tmax_mth", np.empty((1, NY, NX), np.float64)),
                     ("tmin_mth", None), ("tmax", np.empty((nd, NY, NX), np.float32))):
        out = days_out(nd, 1)
        out[key] = bad
        with pytest.raises(ValueError):
            cx.tile_days_mth(ctx(), ctx(), nd, (NY, NX), g, out=out)
    out = days_out(nd, 1)
    out["tmin_mth"] = fake_device(out["tmin_mth"])
    with pytest.raises(ValueError, match="same memory space"):
        cx.tile_days_mth(ctx(), ctx(), nd, (NY, NX), g, out=out)
    for kw in (dict(), dict(out=days_out(nd, 1))):
        with pytest.raises(TwxiError):
            cx.tile_days_mth(ctx(), ctx(), nd, (NY, NX), g, **kw)
    with pytest.raises(TwxiError):                            # a window that completes no month
        cx.tile_days_mth(ctx(), ctx(), 10, (NY, NX), g, out=days_out(10, 0))
    assert g.day0 == 0                                        # a failed call does not advance the groups


def test_tile_end_checks(cx, TwxiError):
    for key, bad in (("tmin_norm", None), ("tmax_se", np.empty((12, NY, NX), np.float64)),
                     ("ninvalid", np.empty((NX, NY), np.int32)), ("status", np.empty((NY, NX), np.int8))):
        out = end_out()
        out[key] = bad
        with pytest.raises(ValueError):
            cx.tile_end(ctx(), ctx(), (NY, NX), out=out)
    out = end_out()
    out["status"] = fake_device(out["status"])
    with pytest.raises(ValueError, match="same memory space as the other result buffers"):
        cx.tile_end(ctx(), ctx(), (NY, NX), out=out)
    for kw in (dict(), dict(out=end_out())):
        with pytest.raises(TwxiError):
            cx.tile_end(ctx(), ctx(), (NY, NX), **kw)

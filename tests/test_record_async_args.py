"""Argument checks of the asynchronous tile wrappers in context.py (CPU only): with host buffers, wait=False needs the
caller's ``out`` and pinned torch tensors, and says so before any library call.

The library is replaced by a stub that fails the test on any attribute access, so a check that came after the call would
show up as an AssertionError instead of the ValueError."""
import types

import numpy as np
import pytest

NY, NX, ND = 3, 4, 40


class NoLibrary(object):
    def __getattr__(self, name):
        raise AssertionError("library entry point %s reached before the argument check" % name)


@pytest.fixture()
def cx(monkeypatch):
    from topowx_b200 import build
    build.build_lib()
    from topowx_b200 import context
    monkeypatch.setattr(context, "lib", NoLibrary())
    return context


def ctx(ndays=ND):
    return types.SimpleNamespace(ndays=ndays, handle=None)


def fin_out(mk):
    return dict(tmin_norm=mk((12, NY, NX), "float32"), tmax_norm=mk((12, NY, NX), "float32"),
                tmin_se=mk((12, NY, NX), "float32"), tmax_se=mk((12, NY, NX), "float32"),
                ninvalid=mk((NY, NX), "int32"), status=mk((NY, NX), "uint8"))


def test_host_buffers_without_out_are_refused(cx):
    from topowx_b200 import synth
    with pytest.raises(ValueError, match="needs `out`"):
        cx.tile_days(ctx(), ctx(), 5, (NY, NX), wait=False)
    groups = cx.MonthGroups(synth.make_days(1995, 1))
    with pytest.raises(ValueError, match="needs `out`"):
        cx.tile_days_mth(ctx(), ctx(), 5, (NY, NX), groups, wait=False)
    assert groups.day0 == 0                                           # the month runs did not advance
    with pytest.raises(ValueError, match="needs `out`"):
        cx.tile_end(ctx(), ctx(), (NY, NX), wait=False)


def test_unpinned_torch_buffers_are_refused(cx):
    import torch
    mk = lambda shape, dt: torch.empty(shape, dtype=getattr(torch, dt))
    with pytest.raises(ValueError, match="not pinned"):
        cx.tile_days(ctx(), ctx(), 5, (NY, NX), out=dict(tmin=mk((5, NY, NX), "int16"), tmax=mk((5, NY, NX), "int16")),
                     wait=False)
    with pytest.raises(ValueError, match="not pinned"):
        cx.tile_end(ctx(), ctx(), (NY, NX), out=fin_out(mk), wait=False)
    with pytest.raises(ValueError, match="not pinned"):
        cx.tile_begin(ctx(), ctx(), torch.zeros((32, NY, NX), dtype=torch.float64), wait=False)


def test_waiting_calls_keep_their_allocation(cx):
    """wait=True still allocates host buffers itself: it reaches the (stubbed) library."""
    with pytest.raises(AssertionError, match="twxi_tile_days reached"):
        cx.tile_days(ctx(), ctx(), 5, (NY, NX))
    with pytest.raises(AssertionError, match="twxi_tile_days_async reached"):
        cx.tile_days(ctx(), ctx(), 5, (NY, NX), out=dict(tmin=np.empty((5, NY, NX), np.int16),
                                                          tmax=np.empty((5, NY, NX), np.int16)), wait=False)

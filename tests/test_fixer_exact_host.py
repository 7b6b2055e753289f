"""The exact referee of the Tmin >= Tmax fixer stage, and the proof that it is sharp.  CPU only.

The fixer (fix_inverted in csrc/twxi_internal.cuh, run by fixer_kernel over the whole record and by tile_fix_kernel over
day windows) is bookkeeping, not numerics: which days are fixed, which 31-day window each fix reads, and that days fixed
earlier feed the windows of later fixes.  The referee below judges one fix at a time against exact rational arithmetic on
the state the device itself saw at that fix (its own final values before the day, the unfixed values from the day on), so
rounding cannot accumulate and any wrong window, wrong validity test or wrong read order shows up by orders of magnitude
above the bound.  The same module judges the recomputed 1981-2010 normals and the int16 quantisation.

tests/test_gpu_fixer_exact.py applies these checks to the device's dailies.  Here they are held to the reference's own
code (the golden vectors of tests/golden/tmin_tmax_fixer.npz and the oracle), and every seeded defect of a numpy copy of
the device fixer, on the crafted inversion patterns the GPU test uses, must be rejected while the faithful copy passes."""
from fractions import Fraction

import numpy as np
import pytest

from oracle import twx_oracle as o

EPS = 2.0 ** -53                        # unit roundoff of float64
TAIL = 15                               # half-window of the fixer (interp_tair.py:177-183)
ST_OK, ST_FIXER_EMPTY = 0, 5
FILL_I2, FILL_I4, FILL_F4, FILL_F8 = -32767, -2147483647, np.float32(9.969209968386869e+36), 9.969209968386869e+36


# ---- crafted inversion patterns ---------------------------------------------------------------------------------------
def delta_pattern(nd, inverted=(), tied=()):
    """Tmax - Tmin per day: -2 on `inverted` days, exactly 0 on `tied` days (an inversion, since the fixer tests >=), and
    2 + 0.1 (d mod 7) on every valid day, so a window that is one day long or short changes the mean it reads."""
    d = np.arange(nd)
    delta = 2.0 + 0.1 * (d % 7)
    delta[np.asarray(inverted, dtype=np.int64)] = -2.0
    delta[np.asarray(tied, dtype=np.int64)] = 0.0
    return delta


def smooth_anomaly(nd):
    """A smooth per-day anomaly (C) shared by Tmin and Tmax."""
    d = np.arange(nd, dtype=np.float64)
    return 3.0 * np.sin(2 * np.pi * d / 365.25) + 1.5 * np.sin(2 * np.pi * d / 23.0 + 0.4)


# The patterns of the crafted records (first day, number of days, inverted days, tied days).  The GPU test builds twin
# station tables that reproduce them in every cell; the CPU tests below apply them to plain series.
def _span(a, b):
    return list(range(a, b))


CRAFTED = {
    # 1995: a run at days 0..14 fixed from day 15 (a tie inside it), isolated inversions at x = 31, 0, 1 (mod 32) across
    # ballot passes, ties, a 50-day run across the 16/31/32/33-day window boundaries and two ballot passes, and the last
    # 15 days (windows clipped at the end)
    "y1995": ((1995, 1, 1), 365, _span(0, 7) + _span(8, 15) + [31, 32, 33, 63, 96, 129] + _span(150, 200) + _span(350, 365),
              [7, 40, 41, 250, 251, 252]),
    # 1980-07-01 .. 1982-06-30: the 1981-2010 groups start mid-record (1981-01-01 is day 184, inside a run), months 7-12
    # of 1982 are empty groups (NaN normals in fixed cells); the last 8 days are inverted and the 7 before them valid, so
    # a window of day 0 that wrapped around to the record end would read valid days
    "rec1980": ((1980, 7, 1), 730, _span(0, 10) + _span(175, 200) + [287, 288, 289] + _span(440, 490) + _span(722, 730),
                [300, 301, 500, 191]),
    # days 0..15 inverted: the fix of day 0 finds no valid day ('No valid tmin/tmax in window') in every cell
    "empty_start": ((1995, 1, 1), 60, [d for d in range(16) if d != 5], [5]),
    # every day tied: every cell fails at day 0
    "all_tied": ((1995, 1, 1), 40, [], _span(0, 40)),
    # short records from 1995-01-01 (one January; one ballot pass, exactly one, one and a day)
    "short20": ((1995, 1, 1), 20, _span(0, 15), []),
    "short31": ((1995, 1, 1), 31, _span(0, 5) + _span(16, 31), [10]),
    "short32": ((1995, 1, 1), 32, _span(0, 5) + _span(17, 32), [10, 31]),
    "short33": ((1995, 1, 1), 33, _span(0, 5) + _span(18, 33), [10, 32]),
}


def crafted_days(name):
    from datetime import datetime, timedelta
    from topowx_b200 import db
    (y, m, d), nd, _, _ = CRAFTED[name]
    t0 = datetime(y, m, d)
    return db.get_days_metadata(t0, t0 + timedelta(days=nd - 1))


def crafted_delta(name):
    _, nd, inv, tie = CRAFTED[name]
    return delta_pattern(nd, inv, tie)


# ---- the referee --------------------------------------------------------------------------------------------------------
def _F(x):
    return Fraction(float(x))


def fix_bound(tavg, half):
    """Bound on |device - exact| of one fixed value tavg -/+ half, given exact inputs (the device's own state).

    The device forms each valid diff hi - lo (one rounding), sums at most 31 of them in a five-level shuffle tree (five
    roundings on a sum of positive terms), divides by the count (one) and by 2 (exact): the computed half is within
    (1 + u)^7 - 1 < 7.01 u of |half| relative, u = 2^-53, because every term is positive.  tavg = (tmin + tmax) / 2 is one
    rounding (u |tavg|), and tavg -/+ half one more (u (|tavg| + half)).  Together: 2 u |tavg| + 8.01 u half, below
    8 u (|tavg| + half) with room for the second-order terms.  A window one day off moves the value by ~(spread of the
    diffs) / 31, i.e. >= 1e-3 C on the crafted patterns, twelve orders above the bound."""
    return 8 * EPS * (abs(tavg) + half)


def oracle_status(tmin0, tmax0):
    """TWXI_ST_FIXER_EMPTY when oracle.tmin_tmax_fixer on the unfixed series finds a window without a valid day.  A fixed day
    is always valid, so the float64 oracle takes every validity decision exactly as the device does."""
    try:
        o.tmin_tmax_fixer(np.asarray(tmin0, dtype=np.float64), np.asarray(tmax0, dtype=np.float64))
    except o.OracleError as e:
        assert e.status == ST_FIXER_EMPTY
        return ST_FIXER_EMPTY
    return ST_OK


def _same_bits(a, b):
    return np.array_equal(np.asarray(a, dtype=np.float64).view(np.int64), np.asarray(b, dtype=np.float64).view(np.int64))


def check_fixes(tmin0, tmax0, tmin1, tmax1, ninvalid):
    """One cell whose fixer succeeded: (tmin0, tmax0) unfixed, (tmin1, tmax1) fixed by the implementation under test,
    ninvalid its count.  The fixed days are exactly nonzero(tmin0 >= tmax0), every other day keeps its bits, and each fix x
    is tavg -/+ the mean valid diff over days max(x-15, 0) .. min(x+15, nd-1) in exact arithmetic, read from the final
    values of days < x and the unfixed values of days >= x, within fix_bound.  Returns (fixed days, largest error / bound);
    raises AssertionError at the first violation."""
    tmin0, tmax0 = np.asarray(tmin0, dtype=np.float64), np.asarray(tmax0, dtype=np.float64)
    tmin1, tmax1 = np.asarray(tmin1, dtype=np.float64), np.asarray(tmax1, dtype=np.float64)
    nd = tmin0.size
    inv = np.flatnonzero(tmin0 >= tmax0)
    assert int(ninvalid) == inv.size, "ninvalid %d, %d days with tmin >= tmax" % (int(ninvalid), inv.size)
    keep = np.ones(nd, dtype=bool)
    keep[inv] = False
    assert _same_bits(tmin1[keep], tmin0[keep]) and _same_bits(tmax1[keep], tmax0[keep]), \
        "a day without tmin >= tmax changed: %s" % np.flatnonzero(keep & ((tmin1 != tmin0) | (tmax1 != tmax0)))[:8]
    worst = 0.0
    for x in inv:
        s, e = max(x - TAIL, 0), min(x + TAIL + 1, nd)
        before = np.arange(s, e) < x
        lo = np.where(before, tmin1[s:e], tmin0[s:e])
        hi = np.where(before, tmax1[s:e], tmax0[s:e])
        ok = lo < hi
        assert ok.any(), "day %d: no valid day in its window, but the fix succeeded" % x
        half = sum(_F(h) - _F(l) for h, l in zip(hi[ok], lo[ok])) / (2 * int(ok.sum()))
        tavg = (_F(tmin0[x]) + _F(tmax0[x])) / 2
        bound = fix_bound(float(tavg), float(half))
        for got, want, what in ((tmin1[x], tavg - half, "tmin"), (tmax1[x], tavg + half, "tmax")):
            err = abs(float(_F(got) - want)) if np.isfinite(got) else np.inf
            assert err <= bound, "day %d %s: %r, exact %.17g, error %.3g > bound %.3g" % (x, what, got, float(want), err,
                                                                                         bound)
            worst = max(worst, err / bound)
    return inv, worst


def check_against_oracle(tmin0, tmax0, tmin1, tmax1):
    """The second referee: oracle.tmin_tmax_fixer in float64 on the unfixed series.  Device and oracle each round every
    fix within fix_bound of its exact value on its own state; a fixed day's difference then reaches the later fixes of its
    chain (fixes at most 15 days apart) only through the window mean, with weight <= 1 (fixed days are valid, so they are
    counted).  So the difference at the j-th fix of a chain is at most the sum of 2 fix_bound over fixes 0..j of it."""
    a, b, n = o.tmin_tmax_fixer(np.asarray(tmin0, dtype=np.float64), np.asarray(tmax0, dtype=np.float64))
    inv = np.flatnonzero(np.asarray(tmin0) >= np.asarray(tmax0))
    acc, prev = 0.0, None
    for x in inv:
        if prev is None or x - prev > TAIL:
            acc = 0.0
        prev = x
        acc += 2 * fix_bound(0.5 * abs(a[x] + b[x]), 0.5 * abs(b[x] - a[x]))
        for got, want, what in ((tmin1[x], a[x], "tmin"), (tmax1[x], b[x], "tmax")):
            assert abs(got - want) <= acc, "day %d %s: %r, oracle %r, chain bound %.3g" % (x, what, got, want, acc)
    return n


def normal_groups(days):
    """The 1981-2010 (year, month) groups of a chronological days table as twxi_ctx_set_obs forms them: start and length,
    year-major over the years y0..y1 of the record inside 1981-2010."""
    year, month = np.asarray(days["YEAR"]), np.asarray(days["MONTH"])
    yrs = year[(year >= 1981) & (year <= 2010)]
    y0, y1 = int(yrs.min()), int(yrs.max())
    nyr = y1 - y0 + 1
    gs, gl = np.zeros(nyr * 12, dtype=np.int64), np.zeros(nyr * 12, dtype=np.int64)
    for d in np.flatnonzero((year >= 1981) & (year <= 2010)):
        g = (year[d] - y0) * 12 + month[d] - 1
        if gl[g] == 0:
            gs[g] = d
        gl[g] += 1
    return gs, gl


def normals_bound(vals, lens, nyr):
    """Bound on the recomputed normal of one month: each group mean is a lane-strided sum (len/32 sequential additions),
    a five-level tree and a division; the mean over years adds nyr roundings.  Every term is at most max|t|:
    (len/32 + 8 + nyr) 2 u max|t|."""
    return (max(lens) / 32.0 + 8 + nyr) * 2 * EPS * max(np.abs(vals).max(), 1.0)


def check_normals(t1, gs, gl, nrm):
    """Normals of a cell with ninvalid > 0: the exact mean over years of the monthly means of the fixed days t1 of the
    1981-2010 groups (gs, gl); a month with an empty group is NaN, as np.mean of an empty slice.  Returns the number of
    NaN months."""
    t1 = np.asarray(t1, dtype=np.float64)
    nyr = gl.size // 12
    nnan = 0
    for m in range(12):
        g = [y * 12 + m for y in range(nyr)]
        if any(gl[i] == 0 for i in g):
            assert np.isnan(nrm[m]), "month %d has an empty group: normal %r, not NaN" % (m + 1, nrm[m])
            nnan += 1
            continue
        exact = sum(sum(_F(v) for v in t1[gs[i]:gs[i] + gl[i]]) / int(gl[i]) for i in g) / nyr
        vals = np.concatenate([t1[gs[i]:gs[i] + gl[i]] for i in g])
        bound = normals_bound(vals, [gl[i] for i in g], nyr)
        err = abs(float(_F(nrm[m]) - exact)) if np.isfinite(nrm[m]) else np.inf
        assert err <= bound, "month %d normal %r, exact %.17g, error %.3g > bound %.3g" % (m + 1, nrm[m], float(exact),
                                                                                            err, bound)
    return nnan


def check_quantized(q, f8):
    """int16 dailies against step25's quantisation of the f8 dailies, byte for byte."""
    want = o.quantize_daily(np.asarray(f8, dtype=np.float64))
    bad = np.flatnonzero(np.asarray(q) != want)
    assert bad.size == 0, "int16 dailies differ on %d days, first %d: %d, want %d (from %r)" % (
        bad.size, bad[0], q[bad[0]], want[bad[0]], f8[bad[0]])


# ---- a numpy copy of the device stage, with seeded defects --------------------------------------------------------------
def emulate_fixer(tmin0, tmax0, lo_off=-TAIL, hi_off=TAIL, strict=False, read_unfixed=False, clip=True):
    """fix_inverted in numpy: defaults are the device's arithmetic.  lo_off / hi_off: the window x+lo_off .. x+hi_off;
    strict: `>` instead of `>=`; read_unfixed: windows read the unfixed copy of earlier fixed days; clip=False: days before
    the record start wrap around to its end (negative numpy indices).  Returns (tmin, tmax, ninvalid, status)."""
    tmin, tmax = np.array(tmin0, dtype=np.float64), np.array(tmax0, dtype=np.float64)
    inv = np.flatnonzero(tmin > tmax if strict else tmin >= tmax)
    nd = tmin.size
    for x in inv:
        idx = np.arange(x + lo_off, x + hi_off + 1)
        idx = idx[idx < nd]
        if clip:
            idx = idx[idx >= 0]
        lo = (tmin0 if read_unfixed else tmin)[idx]
        hi = (tmax0 if read_unfixed else tmax)[idx]
        ok = lo < hi
        if not ok.any():
            return None, None, inv.size, ST_FIXER_EMPTY
        half = np.sum(hi[ok] - lo[ok]) / ok.sum() / 2.0
        tavg = (tmin[x] + tmax[x]) / 2.0
        tmin[x], tmax[x] = tavg - half, tavg + half
    return tmin, tmax, inv.size, ST_OK


def emulate_normals(t, gs, gl, short_group=None):
    """fixer_kernel's normals: mean over years of the group means.  short_group: that group loses its last day."""
    nyr = gl.size // 12
    out = np.empty(12)
    with np.errstate(all="ignore"):
        for m in range(12):
            acc = 0.0
            for y in range(nyr):
                g = y * 12 + m
                n = gl[g] - (1 if g == short_group else 0)
                acc += np.sum(t[gs[g]:gs[g] + n]) / n                 # n == 0: NaN, as np.mean of an empty slice
            out[m] = acc / nyr
    return out


def emulate_quantize(x, f32_scale=True):
    """quantize() of twxi_internal.cuh; f32_scale=False divides by the double 0.01 instead of float32(0.01)."""
    r = np.rint(np.asarray(x) * 100.0) / 100.0
    return (r / (np.float64(np.float32(0.01)) if f32_scale else 0.01)).astype(np.int64).astype(np.int16)


def _series(name):
    """A plain cell series with the crafted pattern of `name`: a seasonal Tmin, Tmax = Tmin + delta (ties exactly equal)."""
    days = crafted_days(name)
    nd = days.size
    d = np.arange(nd, dtype=np.float64)
    tmin0 = 4.0 + 9.0 * np.sin(2 * np.pi * (d - 100) / 365.25) + smooth_anomaly(nd)
    delta = crafted_delta(name)
    tmax0 = tmin0 + delta
    tmax0[delta == 0] = tmin0[delta == 0]
    return days, tmin0, tmax0


def _judge(days, tmin0, tmax0, fixed, normals_fn=emulate_normals, quantize_fn=emulate_quantize):
    """Every referee check of one cell on an emulated stage: fixes, oracle, normals, quantisation."""
    tmin1, tmax1, ninv, st = fixed
    want = oracle_status(tmin0, tmax0)
    assert st == want, "status %d, the oracle decides %d" % (st, want)
    if st != ST_OK:
        return
    check_fixes(tmin0, tmax0, tmin1, tmax1, ninv)
    check_against_oracle(tmin0, tmax0, tmin1, tmax1)
    gs, gl = normal_groups(days)
    for t in (tmin1, tmax1):
        check_normals(t, gs, gl, normals_fn(t, gs, gl))
        check_quantized(quantize_fn(t), t)


DEFECTS = {
    "window of 30 days (x-15 .. x+14)": dict(fixer=dict(hi_off=TAIL - 1)),
    "window of 32 days (x-15 .. x+16)": dict(fixer=dict(hi_off=TAIL + 1)),
    "window of 32 days (x-16 .. x+15)": dict(fixer=dict(lo_off=-TAIL - 1)),
    "tmin > tmax instead of >= (ties left unfixed)": dict(fixer=dict(strict=True)),
    "earlier fixed days read unfixed": dict(fixer=dict(read_unfixed=True)),
    # in y1995 the days a wrapped window reads are the inverted last 15 days, which it skips either way
    "window of day 0 not clipped (wraps to the record end)": dict(fixer=dict(clip=False), patterns=("rec1980",)),
    "quantised with / 0.01 instead of / float32(0.01)": dict(quantize=lambda x: emulate_quantize(x, f32_scale=False)),
    "a 1981-2010 group one day short": dict(normals=lambda t, gs, gl: emulate_normals(t, gs, gl, int(np.argmax(gl > 0)))),
}
DEFECT_PATTERNS = ("y1995", "rec1980")


def test_referee_reproduces_the_golden_fixer():
    """The reference's own tmin_tmax_fixer outputs (tests/golden) pass both referees, with their counts."""
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "tmin_tmax_fixer.npz"))
    nfix = 0
    for c in range(5):
        a0, b0 = g["tmin%d" % c], g["tmax%d" % c]
        assert oracle_status(a0, b0) == ST_OK
        inv, worst = check_fixes(a0, b0, g["otmin%d" % c], g["otmax%d" % c], int(g["ninv%d" % c]))
        check_against_oracle(a0, b0, g["otmin%d" % c], g["otmax%d" % c])
        assert worst <= 1.0
        nfix += inv.size
    assert nfix > 20


@pytest.mark.parametrize("name", sorted(CRAFTED))
def test_referee_agrees_with_the_oracle_and_the_faithful_copy(name):
    """On every crafted pattern the oracle's fixed series and the faithful numpy copy of the device stage pass; the
    patterns fail where they are meant to."""
    days, tmin0, tmax0 = _series(name)
    _judge(days, tmin0, tmax0, emulate_fixer(tmin0, tmax0))
    st = oracle_status(tmin0, tmax0)
    assert (st == ST_FIXER_EMPTY) == (name in ("empty_start", "all_tied"))
    if st == ST_OK:
        a, b, n = o.tmin_tmax_fixer(tmin0, tmax0)
        check_fixes(tmin0, tmax0, a, b, n)


@pytest.mark.parametrize("defect", sorted(DEFECTS))
def test_seeded_defect_is_rejected(defect):
    """Each defect of the numpy copy, on the crafted 1995 and 1980-1982 patterns, fails the referee with its bound."""
    spec = DEFECTS[defect]
    msgs = []
    for name in spec.get("patterns", DEFECT_PATTERNS):
        days, tmin0, tmax0 = _series(name)
        fixed = emulate_fixer(tmin0, tmax0, **spec.get("fixer", {}))
        with pytest.raises(AssertionError) as e:
            _judge(days, tmin0, tmax0, fixed, normals_fn=spec.get("normals", emulate_normals),
                   quantize_fn=spec.get("quantize", emulate_quantize))
        msgs.append("%s: %s" % (name, str(e.value).splitlines()[0][:110]))
    print("rejected: %s\n  %s" % (defect, "\n  ".join(msgs)))

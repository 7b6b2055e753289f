"""knn_kernel / knn_candidates_kernel (twxi_knn and the gridded search of twxi_interp_chunk) and nngh_params_kernel
(twxi_nngh_params) held to their contract.

The neighbour search returns the first k+1 stations of the order (km, station index), km as the kernel computes it
(argsort(kind='stable') of the distance vector).  Most of that contract does not depend on device math and is checked
bit for bit:
  1. order: distances non-decreasing, equal distances in ascending station index;
  2. prefix: knn(k) is the first k+1 entries of knn(255), indices and distances, for every k;
  3. leave-outs: rm_idx (1-4 entries, duplicates, -1, stations far away) and rm_zero give the leave-out-free order with
     those stations deleted;
  4. path independence: the fast path (<= 256 candidates), the general path (rank counting), the bitonic sort
     (257-512 keys at or below the threshold) and the pruned gridded search (with and without overflowing candidate
     lists) agree byte for byte;
  5. weights: wgt == (1 - (d / d_bw)^2)^2 evaluated in numpy from the returned d.
What depends on device math is held to ``hav_exact``, the haversine of util_geo.py at 40 digits from the kernel's own
float64 inputs, within C_D u relative (u = 2^-53); no omitted station may be nearer by hav_exact than a returned one by
more than twice that.

Ring fixtures (stations on a circle around the query) put their haversine keys within a few hundred ulps, where
adjacent keys often round to one km: a selection on the haversine key instead of km breaks invariant 2 there.

nngh_params_kernel: TWXI_ST_NO_NNGHS and TWXI_ST_NO_VARIO, smoothed variogram triples within a first-order bound of
their 40-digit weighted means, smoothed counts equal to round-half-even of the 40-digit weighted mean wherever that mean
is farther than its bound from a half-integer, and an exact half-integer mean that must round to even.

Out of scope: the order of numpy's libm at near ties (its keys are not the device's), NaN coordinates, poles and the
antimeridian.

Run with -m gpu; the reference, the fixtures' properties and the (km, index) reference run on the CPU."""
import ctypes as C

import numpy as np
import pytest

mpmath = pytest.importorskip("mpmath")      # comes with torch (through sympy)

DPS = 40
EPS = 2.0 ** -53
RAD = 0.017453292519943295                  # TWX_RAD
R_KM = 6371.009                             # TWX_EARTH_KM
# Relative error of the device's haversine km against hav_exact, in units of u.  CUDA documents sin, cos and asin to
# 2 ulp (<= 4u relative) and sqrt as correctly rounded; the radian products are the kernel's own inputs.  First order:
# sin(dlat/2)^2 and sin(dlon/2)^2 carry 2 (4u + u) + u = 11u with the subtraction, cos(lat1) cos(lat2) 9u, their
# product 21u, the sum a of non-negative terms 22u; sqrt halves that and adds u (12u), asin (condition <= 1.02 below
# 3 000 km) adds 4u, the products by 2 and by R another u: 17.3u.  C_D = 24 leaves the second-order terms room.
C_D = 24
LAT0, LON0 = 40.5, -99.0
K1MAX = 256                                 # TWXI_MAX_NNGHS + 1
MAX_STNS = 24000                            # TWXI_MAX_STNS
ST_OK, ST_NO_NNGHS, ST_NO_VARIO, ST_TOO_FEW, ST_TIES = 0, 1, 2, 3, 7
INIT = 100                                  # TWXI_INIT_NNGHS
OUT_KEYS = ("tmin_norm", "tmax_norm", "tmin_se", "tmax_se", "ninvalid", "status")


# ---- the reference --------------------------------------------------------------------------------------------------
def host_keys(lat0, lon0, lat, lon):
    """The haversine "a" term in the kernel's operation order (hav_a), numpy float64."""
    l1, o1 = lat0 * RAD, lon0 * RAD
    l2, o2 = np.asarray(lat) * RAD, np.asarray(lon) * RAD
    s1, s2 = np.sin((l1 - l2) / 2), np.sin((o1 - o2) / 2)
    return s1 * s1 + (np.cos(l1) * np.cos(l2)) * (s2 * s2)


def host_km(a):
    return R_KM * (2.0 * np.arcsin(np.sqrt(a)))


def hav_exact(lat0, lon0, lat, lon):
    """util_geo.py's haversine km at DPS digits from the kernel's float64 radians fl(lat RAD), fl(lon RAD): everything
    after those products is exact.  Returns an object array of mpf."""
    la2, lo2 = np.asarray(lat, dtype=np.float64) * RAD, np.asarray(lon, dtype=np.float64) * RAD
    with mpmath.workdps(DPS):
        p1, l1 = mpmath.mpf(float(lat0 * RAD)), mpmath.mpf(float(lon0 * RAD))
        c1, R = mpmath.cos(p1), mpmath.mpf(R_KM)
        out = []
        for p2, l2 in zip(la2, lo2):
            p2, l2 = mpmath.mpf(float(p2)), mpmath.mpf(float(l2))
            a = mpmath.sin((p1 - p2) / 2) ** 2 + c1 * mpmath.cos(p2) * mpmath.sin((l1 - l2) / 2) ** 2
            out.append(2 * R * mpmath.asin(mpmath.sqrt(a)))
    return np.array(out, dtype=object)


def topk_km_index(d, k1):
    """The contract on given distances: the first k1 of the order (km, station index)."""
    return np.lexsort((np.arange(d.size), d))[:k1]


def bisquare(d):
    """(1 - (d / d_bw)^2)^2 in numpy float64, d_bw the last distance of each row (station_select.py:169)."""
    r = d / d[..., -1:]
    u = 1.0 - r * r
    return u * u


def ring(n, radius_km, seed, lat0=LAT0, lon0=LON0):
    """n stations at one great-circle distance from (lat0, lon0), random bearings."""
    r = np.random.default_rng(seed)
    th, dd = r.uniform(0, 2 * np.pi, n), radius_km / R_KM
    p0 = lat0 * RAD
    la = np.arcsin(np.sin(p0) * np.cos(dd) + np.cos(p0) * np.sin(dd) * np.cos(th))
    lo = lon0 * RAD + np.arctan2(np.sin(th) * np.sin(dd) * np.cos(p0), np.cos(dd) - np.sin(p0) * np.sin(la))
    return la / RAD, lo / RAD


def scatter(n, rmin_km, rmax_km, seed, lat0=LAT0, lon0=LON0):
    """n stations at random bearings and distances in [rmin_km, rmax_km] (distinct distances)."""
    r = np.random.default_rng(seed)
    lat, lon = [], []
    for d in r.uniform(rmin_km, rmax_km, n):
        a, b = ring(1, d, int(r.integers(1 << 30)), lat0, lon0)
        lat.append(a[0])
        lon.append(b[0])
    return np.array(lat), np.array(lon)


def collapsed_boundaries(lat0, lon0, lat, lon, kmax=K1MAX):
    """k1 values at which a (haversine key, index) selection differs from the (km, index) one, host arithmetic."""
    a = host_keys(lat0, lon0, lat, lon)
    d, i = host_km(a), np.arange(a.size)
    by_key, by_km = np.lexsort((i, a)), np.lexsort((i, d))
    return [k1 for k1 in range(1, min(a.size, kmax) + 1) if set(by_key[:k1]) != set(by_km[:k1])]


class _Stats(object):
    """Worst error / bound ratio per key, and counts."""

    def __init__(self):
        self.d = {}

    def add(self, key, ratio):
        self.d[key] = max(self.d.get(key, 0.0), float(ratio))

    def report(self, title):
        print("\n" + title)
        for key in sorted(self.d):
            print("  %-56s %.3g" % (key, self.d[key]))


STATS = _Stats()


# ---- station tables -------------------------------------------------------------------------------------------------
def make_stns(lat, lon, optim=20.0, optim_anom=20.0, vario=(0.3, 1.0, 60.0)):
    """Station table with the given coordinates (context order = this order); optim, optim_anom and each vario column
    are scalars or per-station arrays, the same for every month."""
    from topowx_b200 import db
    n = len(lat)
    s = np.zeros(n, dtype=db.station_dtype())
    s[db.STN_ID] = ["KNN%06d" % i for i in range(n)]
    s[db.STN_NAME] = s[db.STN_ID]
    s[db.STATE] = "XX"
    s[db.LAT], s[db.LON] = lat, lon
    s[db.ELEV], s[db.TDI], s[db.MASK], s[db.BAD], s[db.CLIMDIV] = 500.0, 0.0, 1.0, np.nan, 1.0
    for m in range(1, 13):
        s[db.get_lst_varname(m)] = 10.0
        s[db.get_norm_varname(m)] = 10.0
        s[db.get_optim_varname(m)] = optim
        s[db.get_optim_anom_varname(m)] = optim_anom
        for p, v in zip((db.VARIO_NUG, db.VARIO_PSILL, db.VARIO_RNG), vario):
            s[db.get_krigparam_varname(m, p)] = v
    return s


def make_ctx(stns):
    from topowx_b200 import db, synth
    from topowx_b200.context import TwxiContext
    days = synth.make_days(1995, 1)[:31]
    da = db.StationSerialDataDb((stns, np.zeros((days.size, stns.size), np.float32), days), "tmin")
    return TwxiContext(da, None, with_obs=False)


def knn(ctx, lat, lon, k, rm_idx=None, rm_zero=False):
    idx, dist, wgt, st = ctx.knn(np.atleast_1d(lat), np.atleast_1d(lon), k, rm_idx=rm_idx, rm_zero=rm_zero)
    return idx, dist, wgt, st


# ---- checks ---------------------------------------------------------------------------------------------------------
def check_order(idx, dist, wgt=None):
    """Invariants 1 and 5 on one row."""
    assert len(set(idx.tolist())) == idx.size
    assert np.all(dist[1:] >= dist[:-1])
    eq = dist[1:] == dist[:-1]
    assert np.all(idx[1:][eq] > idx[:-1][eq]), "equal distances out of station index order"
    if wgt is not None:
        assert np.array_equal(wgt.view(np.uint64), bisquare(dist).view(np.uint64))


def check_exact(key, lat0, lon0, lat, lon, idx, dist, removed=()):
    """Returned distances within C_D u of hav_exact; no omitted, non-removed station nearer than the farthest returned
    one by more than 2 C_D u.  Stations whose host distance exceeds the bandwidth by 1e-9 relative cannot be (the host's
    own error is ~1e-15) and are not evaluated."""
    dh = host_km(host_keys(lat0, lon0, lat, lon))
    out = np.ones(lat.size, dtype=bool)
    out[idx] = False
    out[list(removed)] = False
    cand = np.nonzero(out & (dh <= dist[-1] * (1 + 1e-9)))[0]
    ex_r = hav_exact(lat0, lon0, lat[idx], lon[idx])
    bad = []
    with mpmath.workdps(DPS):
        for j, (d, e) in enumerate(zip(dist, ex_r)):
            err = abs(mpmath.mpf(float(d)) - e)
            if e == 0:
                assert d == 0.0
                continue
            r = float(err / (C_D * EPS * e))
            STATS.add(key + ": distance", r)
            if r > 1:
                bad.append((j, int(idx[j]), float(d), float(e), r))
        far = max(ex_r)
        if cand.size:
            ex_c = hav_exact(lat0, lon0, lat[cand], lon[cand])
            for s, e in zip(cand, ex_c):
                if far > 0:
                    STATS.add(key + ": omitted nearer", float((far - e) / (2 * C_D * EPS * far)))
                if e < far * (1 - 2 * C_D * EPS):
                    bad.append(("omitted", int(s), float(e), float(far)))
    assert not bad, bad[:5]


# ---- CPU: the reference and the fixtures --------------------------------------------------------------------------
def test_hav_exact_matches_the_oracle_distances():
    """hav_exact against the oracle's float64 grt_circle_dist within the host's bound: glibc's sin, cos and asin are
    below 1 ulp, so C_D / 2."""
    from oracle import twx_oracle as o
    lat, lon = scatter(400, 0.5, 2500.0, 11)
    lat, lon = np.concatenate([lat, [LAT0]]), np.concatenate([lon, [LON0]])
    ref = o.grt_circle_dist(LON0, LAT0, lon, lat)
    ex = hav_exact(LAT0, LON0, lat, lon)
    worst = 0.0
    with mpmath.workdps(DPS):
        for d, e in zip(ref, ex):
            if e == 0:
                assert d == 0.0
                continue
            worst = max(worst, float(abs(mpmath.mpf(float(d)) - e) / (EPS * e)))
    assert worst <= C_D / 2, worst
    assert np.array_equal(host_km(host_keys(LAT0, LON0, lat, lon)), ref)     # host_keys is the oracle's arithmetic


def test_km_index_reference_is_prefix_consistent():
    """The (km, index) selection on given distances: knn(k) is the prefix of knn(255) (invariant 2), with many exact
    ties."""
    r = np.random.default_rng(3)
    for trial in range(20):
        d = np.round(r.uniform(1, 50, 600), 1 + trial % 3)          # many exact ties
        full = topk_km_index(d, K1MAX)
        for k1 in range(1, K1MAX + 1):
            assert np.array_equal(topk_km_index(d, k1), full[:k1])
        assert np.all(np.diff(d[full]) >= 0)
        eq = np.diff(d[full]) == 0
        assert np.all(np.diff(full)[eq] > 0)


# name: (stations, radius km, seed, collapsed boundaries the host must find).  250 stations take the fast path, 2 000 the
# general path with rank counting; at 1 500 km 500 stations share 13 distinct km on the host, so about 290 of them lie at
# or below the 256th distance: the bitonic sort orders collapsed keys.  (2 000 stations at 1 500 km put more than 512 at
# or below it on the device: TWXI_ST_KNN_TIES.)
RINGS = {"ring 250 x 150 km": (250, 150.0, 1, 60), "ring 2000 x 150 km": (2000, 150.0, 2, 100),
         "ring 500 x 1500 km": (500, 1500.0, 3, 100)}


@pytest.mark.parametrize("name", sorted(RINGS))
def test_ring_fixture_collapses_key_boundaries(name):
    """On the host, a (key, index) selection differs from the (km, index) one at >= N of the k1 values of each ring."""
    n, rad, seed, need = RINGS[name]
    lat, lon = ring(n, rad, seed)
    a = host_keys(LAT0, LON0, lat, lon)
    assert (a.max() - a.min()) / np.spacing(a.mean()) < 5000          # keys within a few thousand ulps
    bad = collapsed_boundaries(LAT0, LON0, lat, lon)
    assert len(bad) >= need, (name, len(bad))


def cluster_table(c, seed=5, m=200, nfar=30):
    """m scattered stations at 5-30 km, c co-located ones at 60 km, nfar at 300-500 km; the first min(c, 56) cluster
    members are shuffled among the others, the rest appended, so tables that differ in c agree on their common part."""
    lat, lon = scatter(m, 5.0, 30.0, seed)
    fl, fo = scatter(nfar, 300.0, 500.0, seed + 1)
    cl, co = ring(1, 60.0, seed + 2)
    base = np.concatenate([lat, fl, np.repeat(cl, min(c, 56))]), np.concatenate([lon, fo, np.repeat(co, min(c, 56))])
    perm = np.random.default_rng(seed).permutation(base[0].size)
    extra = max(c - 56, 0)
    return (np.concatenate([base[0][perm], np.repeat(cl, extra)]), np.concatenate([base[1][perm], np.repeat(co, extra)]),
            m)


def test_cluster_fixture_counts():
    """The keys at or below the k1 = 256 threshold number exactly m + c (256, 257, 512, 513 for the four tables): the
    cluster lies beyond every scattered station and before every far one."""
    for c in (56, 57, 312, 313):
        lat, lon, m = cluster_table(c)
        d = host_km(host_keys(LAT0, LON0, lat, lon))
        order = topk_km_index(d, lat.size)
        thr = d[order[K1MAX - 1]]
        assert (d <= thr).sum() == m + c
        assert np.unique(d[order[:m]]).size == m and d[order[m - 1]] < thr


def pruning_fixture():
    """A 25 x 25 chunk (one candidate block): k1 stations packed around the block's centre cell, a few stations 2-9 km
    beyond its corner cell (0, 0) on the line from the centre, background stations over 1 degree.  Returns lat, lon of
    the stations, the chunk origin and the cell coordinates."""
    from topowx_b200 import synth
    row0, col0 = synth.TILE_ROW0 + 100, synth.TILE_COL0 + 100
    clat, clon = synth.grid_lats(np.arange(row0, row0 + 25)), synth.grid_lons(np.arange(col0, col0 + 25))
    r = np.random.default_rng(77)
    c_lat, c_lon = clat[12], clon[12]
    lat = [c_lat + r.uniform(-0.002, 0.002, 160)]
    lon = [c_lon + r.uniform(-0.002, 0.002, 160)]
    t = r.uniform(0.15, 0.6, 12)                                    # beyond the corner: (corner - centre) * (1 + t)
    lat.append(clat[0] + (clat[0] - c_lat) * t)
    lon.append(clon[0] + (clon[0] - c_lon) * t)
    lat.append(r.uniform(c_lat - 0.5, c_lat + 0.5, 400))
    lon.append(r.uniform(c_lon - 0.5, c_lon + 0.5, 400))
    return np.concatenate(lat), np.concatenate(lon), (row0, col0), (clat, clon)


def test_pruning_fixture_needs_the_2delta_margin():
    """Some cell's k1 = 101 nearest stations reach beyond r_c + delta of the centre cell (host arithmetic, 1e-6 margin):
    a candidate radius of r_c + delta would drop them."""
    lat, lon, _, (clat, clon) = pruning_fixture()
    k1 = INIT + 1
    dc = host_km(host_keys(clat[12], clon[12], lat, lon))
    rc = np.sort(dc)[k1 - 1]
    la2, lo2 = np.meshgrid(clat, clon, indexing="ij")
    delta = host_km(host_keys(clat[12], clon[12], la2.ravel(), lo2.ravel())).max()
    beyond = 0
    for la, lo in zip(la2.ravel(), lo2.ravel()):
        d = host_km(host_keys(la, lo, lat, lon))
        near = topk_km_index(d, k1)
        beyond = max(beyond, int((dc[near] > (rc + delta) * (1 + 1e-6)).sum()))
    assert beyond >= 3, beyond


# ---- GPU: the search ------------------------------------------------------------------------------------------------
def _queries(lat0=LAT0, lon0=LON0):
    """The centre and three points 0.3-3 km from it."""
    return np.array([lat0, lat0 + 0.01, lat0 - 0.027, lat0 + 0.002]), np.array([lon0, lon0 - 0.004, lon0 + 0.02,
                                                                                 lon0 + 0.03])


def _prefix_and_order(key, ctx, qlat, qlon, kmax, slat, slon):
    """Invariants 1, 2 and 5 for k = 1..kmax, the reference for k = kmax.  Returns knn(kmax)."""
    idx, dist, wgt, st = knn(ctx, qlat, qlon, kmax)
    assert np.all(st == ST_OK)
    for q in range(qlat.size):
        check_order(idx[q], dist[q], wgt[q])
        check_exact(key, qlat[q], qlon[q], slat, slon, idx[q], dist[q])
    bad = []
    for k in range(1, kmax):
        i, d, w, s = knn(ctx, qlat, qlon, k)
        assert np.all(s == ST_OK)
        if not (np.array_equal(i, idx[:, :k + 1]) and np.array_equal(d, dist[:, :k + 1])):
            bad.append(k)
        assert np.array_equal(w.view(np.uint64), bisquare(d).view(np.uint64)), k
    assert not bad, "knn(k) is not a prefix of knn(%d) at k = %s" % (kmax, bad[:10])
    return idx, dist, wgt


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(RINGS))
def test_ring_prefix_order_and_reference(name):
    """Rings: every k is a prefix of the largest, in (km, index) order, within the reference's bounds.  Reports how many
    adjacent returned stations share one km (distinct stations, distinct keys on the host: collapsed boundaries)."""
    n, rad, seed, _ = RINGS[name]
    lat, lon = ring(n, rad, seed)
    ctx = make_ctx(make_stns(lat, lon))
    qlat, qlon = _queries()
    idx, dist, _ = _prefix_and_order(name, ctx, qlat, qlon, min(n - 1, K1MAX - 1), lat, lon)
    coll = int((dist[0, 1:] == dist[0, :-1]).sum())
    STATS.add("%s: equal adjacent km at the centre (count)" % name, coll)
    assert coll > 0                                                 # the device collapses keys too: the test has teeth


@pytest.mark.gpu
def test_fast_and_general_paths_agree_on_rings_and_ties():
    """The same stations searched by the fast path (a table of <= 256) and by the general path (the same table followed
    by far stations): byte-identical for every k.  The tie table holds exact duplicates at several ranks, so for some k
    the tie lies inside the first k+1 (the fast path hands over to the general path) and for others only beyond."""
    lat, lon = ring(250, 150.0, 1)
    slat, slon = scatter(200, 2.0, 40.0, 21)
    dup = [3, 50, 51, 120, 199]                                     # copies of these stations, interleaved
    tlat, tlon = list(slat), list(slon)
    for j, s in enumerate(dup):
        tlat.insert(7 + 30 * j, slat[s])
        tlon.insert(7 + 30 * j, slon[s])
    flat, flon = scatter(40, 400.0, 600.0, 22)
    qlat, qlon = _queries()
    for key, (a, b) in {"ring 250 fast/general": (lat, lon), "ties fast/general": (np.array(tlat), np.array(tlon))}.items():
        fast = make_ctx(make_stns(a, b))
        gen = make_ctx(make_stns(np.concatenate([a, flat]), np.concatenate([b, flon])))
        kmax = a.size - 1
        idx, dist, _ = _prefix_and_order(key, fast, qlat, qlon, kmax, a, b)
        for k in range(1, kmax + 1):
            x, y = knn(fast, qlat, qlon, k), knn(gen, qlat, qlon, k)
            for u, v in zip(x, y):
                assert np.array_equal(u, v), (key, k)
        if key.startswith("ties"):
            eq = (dist[:, 1:] == dist[:, :-1]).sum()
            assert eq >= len(dup)                                   # the duplicates are exact ties on the device


@pytest.mark.gpu
def test_bitonic_and_tie_limit_boundaries():
    """Clusters of co-located stations at the boundary: 256 keys at or below the threshold (rank counting), 257 and 512
    (bitonic sort) and 513 (TWXI_ST_KNN_TIES).  The first three agree byte for byte for every k; 513 agrees where the
    boundary lies before the cluster and reports the tie limit where it lies in it."""
    qlat, qlon = _queries()[0][:1], _queries()[1][:1]
    res = {}
    for c in (56, 57, 312, 313):
        lat, lon, m = cluster_table(c)
        ctx = make_ctx(make_stns(lat, lon))
        res[c] = [knn(ctx, qlat, qlon, k) for k in range(1, K1MAX)]
        if c == 312:
            _prefix_and_order("cluster 512", ctx, qlat, qlon, K1MAX - 1, lat, lon)
    for k in range(1, K1MAX):
        ref = res[56][k - 1]
        assert ref[3][0] == ST_OK
        for c in (57, 312):
            for u, v in zip(ref, res[c][k - 1]):
                assert np.array_equal(u, v), (c, k)
        if k + 1 <= 200:
            for u, v in zip(ref, res[313][k - 1]):
                assert np.array_equal(u, v), (313, k)
        else:
            assert res[313][k - 1][3][0] == ST_TIES, k
    # the cluster members come in station-index order after the 200 scattered stations
    idx, dist = res[56][-1][0][0], res[56][-1][1][0]
    assert np.unique(dist[200:]).size == 1 and np.all(np.diff(idx[200:]) > 0)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [250, 2000])
def test_leave_outs_delete_exactly_the_listed_stations(n):
    """rm_idx rows of 0-4 entries (duplicates, -1 padding, far stations) give the leave-out-free order with those stations
    deleted, indices and distances byte for byte, on the fast (250) and the general (2000) path."""
    lat, lon = ring(n, 150.0, 1 if n == 250 else 2)
    far_lat, far_lon = scatter(4, 800.0, 900.0, 9)
    lat, lon = np.concatenate([lat, far_lat]), np.concatenate([lon, far_lon])
    ctx = make_ctx(make_stns(lat, lon))                             # 254 stations: fast path; 2004: general path
    qlat, qlon = _queries()
    kfull = min(lat.size, K1MAX) - 1
    idx, dist, _, st = knn(ctx, qlat, qlon, kfull)
    assert np.all(st == ST_OK)
    k = 200
    for q in range(qlat.size):
        s = idx[q]
        farst = n                                                   # a station that is not near the point
        rows = np.array([[s[0], -1, -1, -1], [s[5], s[5], s[9], -1], [s[0], s[1], s[2], s[200]],
                         [farst, -1, s[150], farst], [-1, -1, -1, -1], [s[201], s[199], s[198], s[3]]], dtype=np.int32)
        nr = rows.shape[0]
        i, d, w, st2 = knn(ctx, np.repeat(qlat[q], nr), np.repeat(qlon[q], nr), k, rm_idx=rows)
        assert np.all(st2 == ST_OK)
        for r in range(nr):
            keep = ~np.isin(s, rows[r])
            assert np.array_equal(i[r], s[keep][:k + 1]), (q, r)
            assert np.array_equal(d[r], dist[q][keep][:k + 1]), (q, r)
            check_order(i[r], d[r], w[r])


@pytest.mark.gpu
@pytest.mark.parametrize("n", [240, 400])
def test_rm_zero_deletes_exactly_the_stations_at_distance_zero(n):
    """Three stations on the query point and three co-located at another point: rm_zero deletes the three under the
    query, and only them, on the fast (246 stations) and the general path (406)."""
    lat, lon = scatter(n, 1.0, 40.0, 31)
    p_lat, p_lon = lat[17], lon[17]
    lat = np.concatenate([lat[:50], [LAT0, p_lat], lat[50:120], [p_lat, LAT0, LAT0], lat[120:], [p_lat]])
    lon = np.concatenate([lon[:50], [LON0, p_lon], lon[50:120], [p_lon, LON0, LON0], lon[120:], [p_lon]])
    ctx = make_ctx(make_stns(lat, lon))
    k = min(lat.size - 7, K1MAX - 1)
    for ql, qo, nzero in ((LAT0, LON0, 3), (p_lat, p_lon, 4)):
        i0, d0, _, s0 = knn(ctx, ql, qo, k)
        i1, d1, w1, s1 = knn(ctx, ql, qo, k - nzero, rm_zero=True)
        assert s0[0] == ST_OK and s1[0] == ST_OK
        assert (d0[0] == 0).sum() == nzero and np.all(np.diff(i0[0][:nzero]) > 0)
        assert np.array_equal(i1[0], i0[0][nzero:]) and np.array_equal(d1[0], d0[0][nzero:])
        check_order(i1[0], d1[0], w1[0])
        check_exact("rm_zero %d" % n, ql, qo, lat, lon, i1[0], d1[0], removed=i0[0][:nzero])


@pytest.mark.gpu
def test_too_few_stations_after_leave_outs():
    """Stations available after the leave-outs equal to k1: OK; one fewer: TWXI_ST_TOO_FEW_STNS, on the fast path (250
    stations) and the general path (258 stations)."""
    lat, lon = ring(258, 150.0, 4)
    for n in (250, 258):
        ctx = make_ctx(make_stns(lat[:n], lon[:n]))
        idx = knn(ctx, LAT0, LON0, min(n - 1, K1MAX - 1))[0][0]
        for nrm in (1, 2, 3, 4):
            rm = np.array([idx[:nrm].tolist() + [-1] * (4 - nrm)], dtype=np.int32)
            for k1, want in ((n - nrm, ST_OK), (n - nrm + 1, ST_TOO_FEW)):
                if not 2 <= k1 <= K1MAX:
                    continue
                i, d, w, st = knn(ctx, LAT0, LON0, k1 - 1, rm_idx=rm)
                assert st[0] == want, (n, nrm, k1, st[0])
                if want == ST_OK:
                    m = min(k1, idx.size - nrm)
                    assert np.array_equal(i[0][:m], idx[nrm:nrm + m])


@pytest.mark.gpu
def test_table_of_max_stations():
    """TWXI_MAX_STNS stations (a 199 KB key table): four queries against the reference, and prefixes of knn(255)."""
    r = np.random.default_rng(24)
    lat, lon = r.uniform(33.0, 47.0, MAX_STNS), r.uniform(-110.0, -88.0, MAX_STNS)
    ctx = make_ctx(make_stns(lat, lon))
    qlat, qlon = np.array([40.0, 35.5, 44.9, 38.2]), np.array([-99.0, -105.2, -90.3, -95.0])
    idx, dist, wgt, st = knn(ctx, qlat, qlon, K1MAX - 1)
    assert np.all(st == ST_OK)
    for q in range(4):
        check_order(idx[q], dist[q], wgt[q])
        check_exact("24 000 stations", qlat[q], qlon[q], lat, lon, idx[q], dist[q])
    for k in (1, 34, 100, 147, 254):
        i, d, _, _ = knn(ctx, qlat, qlon, k)
        assert np.array_equal(i, idx[:, :k + 1]) and np.array_equal(d, dist[:, :k + 1])


def _pair_ctx(lat, lon, days):
    """Tmin and Tmax contexts of one station table with synthetic observations."""
    from topowx_b200 import db, synth
    from topowx_b200.context import TwxiContext
    r = np.random.default_rng(8)
    stns = make_stns(lat, lon, optim=r.choice([35.0, 52.0, 76.0], lat.size), optim_anom=r.choice([35.0, 63.0], lat.size),
                     vario=(0.3, 1.0, r.uniform(20.0, 200.0, lat.size)))
    f = synth.Fields()
    stns[db.ELEV] = f.elev(lon, lat)
    for m in range(1, 13):
        stns[db.get_lst_varname(m)] = f.lst(0, m, lon, lat, stns[db.ELEV])
        stns[db.get_norm_varname(m)] = f.tair_norm(0, m, lon, lat, stns[db.ELEV], stns[db.get_lst_varname(m)]) \
            + r.normal(0, 0.3, lat.size)
    obs = synth.make_obs(0, stns, days)
    ctx = []
    for w in (0, 1):
        da = db.StationSerialDataDb((stns, obs + w, days), ("tmin", "tmax")[w])
        ctx.append(TwxiContext(da, None))
    return ctx


def _chunk_outputs(ctx, wrk):
    from topowx_b200.context import interp_chunk
    return interp_chunk(ctx[0], ctx[1], wrk, daily=False)


def _same(a, b):
    return all(np.array_equal(a[k], b[k]) for k in OUT_KEYS)


@pytest.mark.gpu
def test_pruned_gridded_search_equals_full_scan(monkeypatch):
    """Gridded search over per-block candidate lists against the full-table scan (TWXI_KNN_FULL), all chunk outputs byte
    for byte: the 25 x 25 block whose corner cell needs stations beyond r_c + delta, chunks of 1 x N, N x 1 and 26 x 26,
    and a candidate cap exactly at the block's list length (no overflow) and one below it (the block is searched over
    the whole table by knn_kernel mode 1)."""
    from topowx_b200 import synth
    from topowx_b200._lib import lib, check
    lat, lon, (row0, col0), _ = pruning_fixture()
    days = synth.make_days(1995, 1)[:31]
    ctx = _pair_ctx(lat, lon, days)
    f = synth.Fields()
    chunks = {"25x25": (0, 0, 25, 25), "1x60": (3, -10, 1, 60), "60x1": (-20, 7, 60, 1), "26x26": (-1, -1, 26, 26)}
    for name, (dr, dc, ny, nx) in chunks.items():
        wrk = synth.make_wrk_chk(f, row0 + dr, col0 + dc, ny, nx)
        wrk[2], wrk[7] = 1.0, 1.0                                   # every cell unmasked, in the stations' climdiv
        pruned = _chunk_outputs(ctx, wrk)
        assert np.all(pruned["status"] == ST_OK), name
        if name == "25x25":
            v = C.c_double()
            check(lib.twxi_ctx_stat(ctx[0].handle, 0, C.byref(v)))
            length = int(round(v.value))
            assert length == v.value and 32 < length < lat.size
        monkeypatch.setenv("TWXI_KNN_FULL", "1")
        full = _chunk_outputs(ctx, wrk)
        monkeypatch.delenv("TWXI_KNN_FULL")
        assert _same(pruned, full), name
        if name == "25x25":
            for cap in (length, length - 1):
                monkeypatch.setenv("TWXI_KNN_CAP", str(cap))
                capped = _chunk_outputs(ctx, wrk)
                monkeypatch.delenv("TWXI_KNN_CAP")
                assert _same(capped, full), cap


# ---- GPU: nngh_params_kernel ----------------------------------------------------------------------------------------
def _near_far(n_near, n_far, seed):
    """n_near stations at 1-10 km, n_far at 30-60 km (distinct distances)."""
    a, b = scatter(n_near, 1.0, 10.0, seed)
    c, d = scatter(n_far, 30.0, 60.0, seed + 1)
    return np.concatenate([a, c]), np.concatenate([b, d])


@pytest.mark.gpu
def test_nngh_params_failure_statuses():
    """TWXI_ST_NO_NNGHS when the 100 nearest have no finite optim, and when every finite one sits at the bandwidth
    distance (weight exactly 0: two co-located stations at positions 100 and 101, the lower index first);
    TWXI_ST_NO_VARIO when the k nearest all have NaN nugget."""
    lat, lon = _near_far(100, 60, 41)
    optim = np.where(np.arange(160) < 100, np.nan, 40.0)
    ctx = make_ctx(make_stns(lat, lon, optim=optim, optim_anom=optim))
    kn, ka, vario, st = ctx.nngh_params(LAT0, LON0)
    assert st[0] == ST_NO_NNGHS
    # 99 without optim, then two co-located stations at 20 km, then far ones: the 100th neighbour has weight 0
    a, b = scatter(99, 1.0, 10.0, 42)
    cl, co = ring(1, 20.0, 43)
    c, d = scatter(60, 30.0, 60.0, 44)
    lat, lon = np.concatenate([a[:40], cl, a[40:], cl, c]), np.concatenate([b[:40], co, b[40:], co, d])
    optim = np.full(lat.size, np.nan)
    optim[[40, 100]] = 12.0
    optim[101:] = 40.0
    ctx = make_ctx(make_stns(lat, lon, optim=optim, optim_anom=optim))
    i, dd, _, s = knn(ctx, LAT0, LON0, 100)
    assert s[0] == ST_OK and i[0][99] == 40 and i[0][100] == 100 and dd[0][99] == dd[0][100]
    assert ctx.nngh_params(LAT0, LON0)[3][0] == ST_NO_NNGHS
    # every optim finite, nugget NaN on the 30 nearest: k_norm = 20 finds no variogram
    lat, lon = _near_far(30, 150, 45)
    nug = np.where(np.arange(180) < 30, np.nan, 0.3)
    ctx = make_ctx(make_stns(lat, lon, optim=20.0, optim_anom=20.0, vario=(nug, 1.0, 60.0)))
    assert ctx.nngh_params(LAT0, LON0)[3][0] == ST_NO_VARIO


@pytest.mark.gpu
@pytest.mark.parametrize("v", [10.5, 12.5])
def test_nngh_count_of_an_exact_half_integer_rounds_to_even(v):
    """One finite neighbour with optim v among the 100 nearest: the weighted mean is exactly v (the host confirms
    fl(fl(v w) / w) == v for the device's weight w), and the count is round-half-even(v)."""
    lat, lon = _near_far(100, 60, 51)
    optim = np.where(np.arange(160) >= 100, 30.0, np.nan)
    ctx = make_ctx(make_stns(lat, lon, optim=optim, optim_anom=optim))
    idx, dist, wgt, st = knn(ctx, LAT0, LON0, INIT)
    j = int(idx[0][37])
    optim[j] = v
    ctx = make_ctx(make_stns(lat, lon, optim=optim, optim_anom=optim))
    idx2, dist2, wgt2, _ = knn(ctx, LAT0, LON0, INIT)
    assert np.array_equal(idx2, idx) and np.array_equal(dist2, dist)
    w = wgt[0][37]
    assert w > 0 and (v * w) / w == v
    kn, ka, vario, st = ctx.nngh_params(LAT0, LON0)
    assert st[0] == ST_OK
    assert np.all(kn[0] == int(np.round(v))) and np.all(ka[0] == int(np.round(v)))


@pytest.mark.gpu
def test_nngh_counts_and_variograms_against_40_digit_means():
    """Synthetic station DB, 64 points: each smoothed count equals round-half-even of the 40-digit weighted mean of the
    100 nearest optim values wherever that mean is farther than its bound from a half-integer (how many are not is
    reported); each variogram triple within a first-order bound of its 40-digit weighted mean over the k_norm nearest."""
    from topowx_b200 import synth, db
    from topowx_b200.context import TwxiContext
    f = synth.Fields()
    days = synth.make_days(1995, 1)[:31]
    da = synth.make_station_db(0, 2000, synth.tile_bbox(), f, days)
    mask = np.isnan(da.stns[db.BAD])
    ctx = TwxiContext(da, mask, with_obs=False)
    s = ctx.stns
    r = np.random.default_rng(64)
    lat = synth.grid_lats(synth.TILE_ROW0 + r.integers(0, 250, 64))
    lon = synth.grid_lons(synth.TILE_COL0 + r.integers(0, 250, 64))
    kn, ka, vario, st = ctx.nngh_params(lat, lon)
    idx, dist, _, st2 = knn(ctx, lat, lon, K1MAX - 1)
    assert np.all(st2 == ST_OK)
    band, checked, bad = 0, 0, []
    with mpmath.workdps(DPS):
        for q in range(lat.size):
            if st[q] != ST_OK:
                continue
            w = bisquare(dist[q][:INIT + 1])[:INIT]
            for m in range(12):
                for kind, col, got in (("norm", db.get_optim_varname(m + 1), kn[q, m]),
                                       ("anom", db.get_optim_anom_varname(m + 1), ka[q, m])):
                    v = s[col][idx[q][:INIT]]
                    ok = np.isfinite(v)
                    num = mpmath.fsum(mpmath.mpf(float(a)) * mpmath.mpf(float(b)) for a, b in zip(v[ok], w[ok]))
                    den = mpmath.fsum(mpmath.mpf(float(b)) for b in w[ok])
                    mean = num / den
                    sabs = float(np.abs(v[ok]) @ w[ok]) / float(den)
                    bound = 2 * (INIT + 2) * EPS * (sabs + abs(float(mean)))      # serial sums of 100 products
                    gap = abs(mean - (mpmath.floor(mean) + mpmath.mpf(0.5)))
                    if gap <= bound:
                        band += 1
                        continue
                    checked += 1
                    if got != int(mpmath.nint(mean)):
                        bad.append((q, m, kind, got, float(mean)))
                k = int(kn[q, m])
                wk = bisquare(dist[q][:k + 1])[:k]
                sl = s[idx[q][:k]]
                vals = [sl[db.get_krigparam_varname(m + 1, p)] for p in (db.VARIO_NUG, db.VARIO_PSILL, db.VARIO_RNG)]
                ok = np.isfinite(vals[0])
                den = mpmath.fsum(mpmath.mpf(float(b)) for b in wk[ok])
                depth = -(-k // 32) + 6                             # lane-strided sums, five warp levels, the product
                for p in range(3):
                    x = vals[p][ok]
                    mean = mpmath.fsum(mpmath.mpf(float(a)) * mpmath.mpf(float(b)) for a, b in zip(x, wk[ok])) / den
                    bound = 2 * depth * EPS * (float(np.abs(x) @ wk[ok]) / float(den) + abs(float(mean)))
                    err = abs(mpmath.mpf(float(vario[q, m, p])) - mean)
                    r_ = float(err / bound) if bound > 0 else (np.inf if err > 0 else 0.0)
                    STATS.add("vario %d" % p, r_)
                    if r_ > 1:
                        bad.append((q, m, "vario", p, float(vario[q, m, p]), float(mean)))
    STATS.add("count: means within their bound of a half-integer (count)", band)
    STATS.add("count: means checked (count)", checked)
    assert checked > 1000 and not bad, bad[:5]


@pytest.mark.gpu
def test_zz_report():
    STATS.report("knn / nngh_params: worst error / bound and counts")

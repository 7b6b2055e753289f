// Stage a8-a9: geographically weighted regression of the daily anomalies, one hat row per (point, month),
// applied to every day of that month.  Replaces GwrTairAnom.gwr_mth (twx/interp/interp_tair.py:261-314) and
// _gwr_series (:1099-1146).
//
// For the k_anom nearest stations (bisquare weights w with the (k+1)-th distance as bandwidth,
// station_select.py:164-169) and X = [1, lon, lat, elev, tdi, lstMM]:   z = x0'(X'WX)^-1 X'W, and
//     daily_t = z . (obs_t - norm) + pt_norm = z . obs_t + (pt_norm - z . norm).
// The 6x6 normal equations are accumulated with the predictors centred on the point and scaled (exactly the
// same predictor because the intercept is in X; the reference inverts the uncentred matrix with LAPACK, which
// loses ~5 digits it never needed) as DMMA outer products, solved with the tensor-pipe pivot-tile factorisation of
// the kriging kernel (chol8_inverse_t), and the hat row is kept in shared memory while the warp streams the month's
// days: lanes = days, neighbours gathered from the station-major,
// month-major observation table (coalesced 128 B per neighbour, L2 resident).
// One warp per (point, month); no intermediate hat rows go to HBM unless the caller asks for them.
#include "twxi_internal.cuh"

#ifndef TWXI_GWR_PACKED_MIN_N
#define TWXI_GWR_PACKED_MIN_N 3000      // station tables above this size are gathered as packed 64-byte rows (see gwr_kernel)
#endif
namespace twxi {

constexpr int GWR_THREADS = 256;
constexpr int GWR_WARPS = GWR_THREADS / 32;
constexpr int GWR_MAXK = 256;
#ifndef TWXI_GWR_MINB
#define TWXI_GWR_MINB 4
#endif

struct GwrArgs {
    StnTable st;
    ObsTable ob;
    int npts, k1, single_mth;
    const int32_t* idx;
    const double* dist;
    const int32_t* nn;
    const double *qlon, *qlat, *qelev, *qtdi, *qlst;
    const double* pt_norm;     // [npts][12] kriged normals, or [npts] when pt_norm_single
    int pt_norm_single;
    double* daily;             // [npts][ndays] chronological, or null
    double* out_month;         // [npts][D_m] month order, or null
    int kmax;                  // hat outputs (null = off)
    int32_t* hat_k;
    int32_t* hat_idx;
    double* hat_z;
    int32_t* status;
    // cross validation of the neighbour count (XvalTairAnom.run_xval, optimize.py:505-545): every point is a station of the
    // table (xv_self, left out by the neighbour search), k is fixed, and instead of daily values the kernel returns
    // bias / MAE / r^2 of the interpolated against the station's own anomalies
    int k_fixed;               // > 0: neighbour count of every point (nn is not read)
    const int32_t* xv_self;    // [npts] station index of the point, or null
    double* xv_out;            // [npts][xv_nc][12][3]
    int xv_nc, xv_ci;
    double* hat_off;           // HAT instance: [npts][12] pt_norm - z . norm
};

// HAT: hat rows of every (point, month) to hat_k / hat_off [npts][12] and hat_idx / hat_z [npts][12][kmax], no daily
// values (the day windows of twxi_tile_days apply them).  A separate instance, so that the production kernel carries no
// branch for it: z and the offset are bitwise what the production instance applies to the days.
template <bool XVAL, bool PACKED, bool HAT = false>
__global__ void __launch_bounds__(GWR_THREADS, TWXI_GWR_MINB) gwr_kernel(GwrArgs a) {
    __shared__ __align__(16) double s_z[GWR_WARPS][GWR_MAXK];
    __shared__ __align__(16) int s_off[GWR_WARPS][GWR_MAXK];                // station * ndays: row offset into obsT
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nm = a.single_mth >= 0 ? 1 : 12;
    const long long item = (long long)blockIdx.x * GWR_WARPS + warp;
    if (item >= (long long)a.npts * nm) return;
    // month-major items: the warps of a CTA work on the same month of consecutive (= adjacent) points, whose neighbour
    // sets nearly coincide, so the station predictors and observation lines they gather are shared through L1
    const int q = (int)(item % a.npts);
    const int m = a.single_mth >= 0 ? a.single_mth : (int)(item / a.npts);
    if (a.status[q] != TWXI_ST_OK) return;
    const int k = XVAL ? a.k_fixed : a.nn[(size_t)q * 24 + 12 + m];
    if (k < 1) return;
    const int N = a.st.n;
    const int32_t* idx = a.idx + (size_t)q * a.k1;
    const double* dist = a.dist + (size_t)q * a.k1;
    const double dbw = dist[k];                               // station_select.py:164
    const double lon0 = a.qlon[q], lat0 = a.qlat[q], elev0 = a.qelev[q], tdi0 = a.qtdi[q];
    const double lst0 = a.qlst[(size_t)q * 12 + m];
    const double* lstm = a.st.lst + (size_t)m * N;
    const double* normm = a.st.norm + (size_t)m * N;

    // ---- X'WX on the tensor pipe --------------------------------------------------------------------------
    // Lane (i, kk) = (lane / 4, lane % 4) supplies predictor i of station 4t + kk scaled by sqrt(w) = 1 - (d/dbw)^2
    // (bisquare w = (1 - (d/dbw)^2)^2, station_select.py:169); the same register is the A and the B operand of one
    // DMMA, which adds the four outer products sqrt(w) x (sqrt(w) x)' of those stations to the 8x8 accumulator.
    const int pi = lane >> 2, kk = lane & 3;
    // PACKED: station rows of the month (1, lon, lat, elev, tdi, lst_m, norm_m, 0), so that the eight lanes of one station
    // read one 64-byte row (two sectors) instead of five scattered ones.  Wins once the six separate arrays no longer
    // stay in L1 (10 000 stations: 4.69 -> 4.56 ms per tile); with 2 000 stations the separate arrays are faster
    // (5.1 against 5.5 ms), hence the two instances.
    const double* gxm = a.st.gx + (size_t)m * N * 8;
    const double* src = PACKED ? gxm + pi : a.st.lon;
    double ref = 0.0, scl = 0.0, cst = 0.0;                   // predictor = (src[s] - ref) * scl + cst
    if (pi == 0) { if (PACKED) scl = 1.0; else cst = 1.0; }
    else if (pi == 1) { ref = lon0; scl = 1.0; }
    else if (pi == 2) { if (!PACKED) src = a.st.lat; ref = lat0; scl = 1.0; }
    else if (pi == 3) { if (!PACKED) src = a.st.elev; ref = elev0; scl = 1e-3; }
    else if (pi == 4) { if (!PACKED) src = a.st.tdi; ref = tdi0; scl = 1.0; }
    else if (pi == 5) { if (!PACKED) src = lstm; ref = lst0; scl = 0.1; }
    // stage the neighbour indices and sqrt(w) once per station (coalesced), padded to a multiple of 16 with weight 0
    const int kpad = (k + 15) & ~15;
    const double rdbw = 1.0 / dbw;
    for (int j = lane; j < kpad; j += 32) {
        int sj = 0;
        double uj = 0.0;
        if (j < k) {
            sj = idx[j];
            const double qd = dist[j] * rdbw;                 // dist / dbw: one reciprocal per warp and a correction step
            const double r = fma(fma(-qd, dbw, dist[j]), rdbw, qd);     // instead of a division per neighbour
            uj = __dsub_rn(1.0, __dmul_rn(r, r));
        }
        s_off[warp][j] = sj;
        s_z[warp][j] = uj;
    }
    __syncwarp();
    double2 c0 = make_double2(0.0, 0.0), c1 = c0, c2 = c0, c3 = c0;
    for (int j0 = 0; j0 < kpad; j0 += 16) {
        double v[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int j = j0 + 4 * e + kk;
            v[e] = s_z[warp][j] * fma(src[s_off[warp][j] * (PACKED ? 8 : 1)] - ref, scl, cst);
        }
        dmma(c0, v[0], v[0]); dmma(c1, v[1], v[1]); dmma(c2, v[2], v[2]); dmma(c3, v[3], v[3]);
    }
    double2 A = make_double2((c0.x + c1.x) + (c2.x + c3.x), (c0.y + c1.y) + (c2.y + c3.y));
    if (lane == 4 * 6 + 3) A.x = 1.0;                         // identity padding of rows / columns 6, 7
    if (lane == 4 * 7 + 3) A.y = 1.0;

    // ---- u = (X'WX)^-1 e_0 from the transposed inverse Cholesky factor Z: (X'WX)^-1 = Z Z' ------------------
    double2 z;
    bool ok = chol8_inverse_t<false>(A, z, lane);
    const double r0x = __shfl_sync(0xffffffffu, z.x, kk), r0y = __shfl_sync(0xffffffffu, z.y, kk);   // row 0 of Z
    double part = fma(z.x, r0x, z.y * r0y);
    part += __shfl_xor_sync(0xffffffffu, part, 1);
    part += __shfl_xor_sync(0xffffffffu, part, 2);            // u_i in the four lanes of row i
    double u[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        u[i] = __shfl_sync(0xffffffffu, part, 4 * i);
        ok = ok && isfinite(u[i]);
    }
    if (!ok) {
        if (lane == 0) atomicCAS(a.status + q, TWXI_ST_OK, TWXI_ST_SINGULAR);
        return;
    }

    // ---- hat row z_j = w_j * (x_j . u) and offset pt_norm - z . norm -------------------------------------
    const size_t nd = (size_t)a.ob.ndays;
    double zn = 0.0;
    for (int j = lane; j < k; j += 32) {
        const int s = s_off[warp][j];
        const double uu = s_z[warp][j];
        const double w = __dmul_rn(uu, uu);
        double xu, nrm;
        if (PACKED) {
            const double2* g2 = reinterpret_cast<const double2*>(gxm + (size_t)s * 8);
            const double2 g01 = g2[0], g23 = g2[1], g45 = g2[2], g67 = g2[3];
            xu = u[0] + u[1] * (g01.y - lon0) + u[2] * (g23.x - lat0) + u[3] * ((g23.y - elev0) * 1e-3)
                 + u[4] * (g45.x - tdi0) + u[5] * ((g45.y - lst0) * 0.1);
            nrm = g67.x;
        } else {
            xu = u[0] + u[1] * (a.st.lon[s] - lon0) + u[2] * (a.st.lat[s] - lat0)
                 + u[3] * ((a.st.elev[s] - elev0) * 1e-3) + u[4] * (a.st.tdi[s] - tdi0)
                 + u[5] * ((lstm[s] - lst0) * 0.1);
            nrm = normm[s];
        }
        const double zj = w * xu;
        s_z[warp][j] = zj;
        s_off[warp][j] = s * (int)nd;
        zn += zj * nrm;
        if constexpr (HAT) {
            const size_t o = ((size_t)q * 12 + m) * a.kmax + j;
            a.hat_z[o] = zj;
            a.hat_idx[o] = s;
        } else if (a.hat_z && j < a.kmax) {                   // (device-resident overrides are not scanned on the host)
            a.hat_z[(size_t)q * a.kmax + j] = zj;
            a.hat_idx[(size_t)q * a.kmax + j] = s;
        }
    }
    zn = warp_sum(zn);
    if constexpr (HAT) {
        if (lane == 0) {
            const double ptn = a.pt_norm[(size_t)q * 12 + m];
            a.hat_k[(size_t)q * 12 + m] = k;
            a.hat_off[(size_t)q * 12 + m] = ptn - zn;
        }
        return;
    }
    if (a.hat_k && lane == 0) a.hat_k[q] = k;
    __syncwarp();
    if (!XVAL && !a.daily && !a.out_month) return;

    // ---- daily values: lanes = days of the month, neighbours gathered from the station-major obs table ------------
    const int self = XVAL ? a.xv_self[q] : 0;
    const double ptn = XVAL ? normm[self] : (a.pt_norm_single ? a.pt_norm[q] : a.pt_norm[(size_t)q * 12 + m]);
    const double off = ptn - zn;
    const int p0 = a.ob.moff[m], D = a.ob.moff[m + 1] - p0;
    double sd = 0.0, sad = 0.0, sx = 0.0, sy = 0.0, sxx = 0.0, syy = 0.0, sxy = 0.0;    // xval sums over the days of this lane
    for (int d0 = 0; d0 < D; d0 += 32) {
        const int d = d0 + lane;
        const bool valid = d < D;
        const float* col = a.ob.obsT + p0 + (valid ? d : 0);
        double acc0 = 0.0, acc1 = 0.0, acc2 = 0.0, acc3 = 0.0;
        int j = 0;
        for (; j + 7 < k; j += 8) {                           // eight gathers in flight per pass (same order of the sums)
            const int4 o4 = *reinterpret_cast<const int4*>(&s_off[warp][j]);
            const int4 o8 = *reinterpret_cast<const int4*>(&s_off[warp][j + 4]);
            const float f0 = col[o4.x], f1 = col[o4.y], f2 = col[o4.z], f3 = col[o4.w];
            const float f4 = col[o8.x], f5 = col[o8.y], f6 = col[o8.z], f7 = col[o8.w];
            const double2 za = *reinterpret_cast<const double2*>(&s_z[warp][j]);
            const double2 zb = *reinterpret_cast<const double2*>(&s_z[warp][j + 2]);
            const double2 zc = *reinterpret_cast<const double2*>(&s_z[warp][j + 4]);
            const double2 zd = *reinterpret_cast<const double2*>(&s_z[warp][j + 6]);
            acc0 = fma(za.x, (double)f0, acc0);
            acc1 = fma(za.y, (double)f1, acc1);
            acc2 = fma(zb.x, (double)f2, acc2);
            acc3 = fma(zb.y, (double)f3, acc3);
            acc0 = fma(zc.x, (double)f4, acc0);
            acc1 = fma(zc.y, (double)f5, acc1);
            acc2 = fma(zd.x, (double)f6, acc2);
            acc3 = fma(zd.y, (double)f7, acc3);
        }
        for (; j + 3 < k; j += 4) {                           // four gathers in flight per pass
            const int4 o4 = *reinterpret_cast<const int4*>(&s_off[warp][j]);
            const float f0 = col[o4.x], f1 = col[o4.y], f2 = col[o4.z], f3 = col[o4.w];
            const double2 za = *reinterpret_cast<const double2*>(&s_z[warp][j]);
            const double2 zb = *reinterpret_cast<const double2*>(&s_z[warp][j + 2]);
            acc0 = fma(za.x, (double)f0, acc0);
            acc1 = fma(za.y, (double)f1, acc1);
            acc2 = fma(zb.x, (double)f2, acc2);
            acc3 = fma(zb.y, (double)f3, acc3);
        }
        for (; j < k; ++j) acc0 = fma(s_z[warp][j], (double)col[s_off[warp][j]], acc0);
        const double v = ((acc0 + acc1) + (acc2 + acc3)) + off;
        if (valid) {
            if (!XVAL && a.daily) a.daily[(size_t)q * nd + a.ob.day_of_pos[p0 + d]] = v;
            if (!XVAL && a.out_month) a.out_month[(size_t)q * D + d] = v;
            if (XVAL) {                                       // optimize.py:520-531
                const double x = v - ptn;                                        // interpolated anomaly
                const double y = (double)a.ob.obsT[(size_t)self * nd + p0 + d] - ptn;    // the station's own anomaly
                const double dif = x - y;
                sd += dif; sad += fabs(dif); sx += x; sy += y; sxx += x * x; syy += y * y; sxy += x * y;
            }
        }
    }
    if (XVAL) {
        sd = warp_sum(sd); sad = warp_sum(sad); sx = warp_sum(sx); sy = warp_sum(sy);
        sxx = warp_sum(sxx); syy = warp_sum(syy); sxy = warp_sum(sxy);
        if (lane == 0) {
            const double n = (double)D;
            const double cxy = sxy - sx * sy / n, cxx = sxx - sx * sx / n, cyy = syy - sy * sy / n;
            const double r = cxy / sqrt(cxx * cyy);           // = scipy.stats.linregress(x, y)[2]
            double* o = a.xv_out + (((size_t)q * a.xv_nc + a.xv_ci) * 12 + m) * 3;
            o[0] = sd / n; o[1] = sad / n; o[2] = r * r;
        }
    }
}

static void gwr_fill(GwrArgs& a, Ctx& c, Batch& b, int mth);

// XvalTairAnom: one launch per neighbour count over (point, month) items; the neighbour search has run once with the
// largest count
int launch_gwr_xval(Ctx& c, Batch& b, const int32_t* self, const int32_t* counts_host, int ncounts, double* out) {
    if (b.npts <= 0) return TWXI_OK;
    GwrArgs a;
    gwr_fill(a, c, b, 0);
    a.xv_self = self; a.xv_out = out; a.xv_nc = ncounts;
    const long long items = (long long)b.npts * 12;
    for (int i = 0; i < ncounts; ++i) {
        a.k_fixed = counts_host[i]; a.xv_ci = i;
        const unsigned grid = (unsigned)((items + GWR_WARPS - 1) / GWR_WARPS);
        if (a.st.n > TWXI_GWR_PACKED_MIN_N) gwr_kernel<true, true><<<grid, GWR_THREADS, 0, c.stream>>>(a);
        else gwr_kernel<true, false><<<grid, GWR_THREADS, 0, c.stream>>>(a);
        TWXI_LAUNCH_CHECK();
    }
    return TWXI_OK;
}

static void gwr_fill(GwrArgs& a, Ctx& c, Batch& b, int mth) {
    a.st = c.st; a.ob = c.ob; a.npts = b.npts; a.k1 = b.k1; a.single_mth = mth >= 1 ? mth - 1 : -1;
    a.idx = b.idx; a.dist = b.dist; a.nn = b.nn;
    a.qlon = b.lon; a.qlat = b.lat; a.qelev = b.elev; a.qtdi = b.tdi; a.qlst = b.lst;
    a.pt_norm = b.mean; a.pt_norm_single = 0; a.daily = nullptr; a.out_month = nullptr;
    a.kmax = 0; a.hat_k = nullptr; a.hat_idx = nullptr; a.hat_z = nullptr; a.status = b.status;
    a.k_fixed = 0; a.xv_self = nullptr; a.xv_out = nullptr; a.xv_nc = 0; a.xv_ci = 0; a.hat_off = nullptr;
}

int launch_gwr(Ctx& c, Batch& b, int mth, const double* pt_norm_override, int write_daily, double* out_month,
               int kmax, int32_t* hat_k, int32_t* hat_idx, double* hat_z) {
    if (b.npts <= 0) return TWXI_OK;
    GwrArgs a;
    gwr_fill(a, c, b, mth);
    a.pt_norm = pt_norm_override ? pt_norm_override : b.mean;
    a.pt_norm_single = pt_norm_override != nullptr;
    a.daily = write_daily ? b.daily : nullptr;
    a.out_month = out_month;
    a.kmax = kmax; a.hat_k = hat_k; a.hat_idx = hat_idx; a.hat_z = hat_z;
    const long long items = (long long)b.npts * (mth >= 1 ? 1 : 12);
    const unsigned grid = (unsigned)((items + GWR_WARPS - 1) / GWR_WARPS);
    if (a.st.n > TWXI_GWR_PACKED_MIN_N) gwr_kernel<false, true><<<grid, GWR_THREADS, 0, c.stream>>>(a);
    else gwr_kernel<false, false><<<grid, GWR_THREADS, 0, c.stream>>>(a);
    TWXI_LAUNCH_CHECK();
    return TWXI_OK;
}

int launch_gwr_hat_rows(Ctx& c, Batch& b, int kh, int32_t* hk, int32_t* hidx, double* hz, double* hoff) {
    if (b.npts <= 0) return TWXI_OK;
    GwrArgs a;
    gwr_fill(a, c, b, 0);
    a.kmax = kh; a.hat_k = hk; a.hat_idx = hidx; a.hat_z = hz; a.hat_off = hoff;
    const long long items = (long long)b.npts * 12;
    const unsigned grid = (unsigned)((items + GWR_WARPS - 1) / GWR_WARPS);
    if (a.st.n > TWXI_GWR_PACKED_MIN_N) gwr_kernel<false, true, true><<<grid, GWR_THREADS, 0, c.stream>>>(a);
    else gwr_kernel<false, false, true><<<grid, GWR_THREADS, 0, c.stream>>>(a);
    TWXI_LAUNCH_CHECK();
    return TWXI_OK;
}

}  // namespace twxi

namespace twxi {

// Points of a cross validation are stations of the table itself (the reference passes the station record as `pt`,
// optimize.py:517,590): gather their coordinates / predictors and leave each one out of its own neighbour search.
__global__ void station_points_kernel(StnTable st, int npts, const int32_t* sidx, Batch b) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= npts) return;
    const int s = sidx[q];
    const bool ok = s >= 0 && s < st.n;
    const int t = ok ? s : 0;
    b.lat[q] = st.lat[t]; b.lon[q] = st.lon[t]; b.elev[q] = st.elev[t]; b.tdi[q] = st.tdi[t];
    for (int m = 0; m < 12; ++m) b.lst[(size_t)q * 12 + m] = st.lst[(size_t)m * st.n + t];
    b.rm_idx[q] = ok ? s : -1;
    b.status[q] = ok ? TWXI_ST_OK : TWXI_ST_TOO_FEW_STNS;
}
int launch_station_points(Ctx& c, Batch& b, int npts, const int32_t* sidx) {
    if (npts <= 0) return TWXI_OK;
    station_points_kernel<<<(npts + 255) / 256, 256, 0, c.stream>>>(c.st, npts, sidx, b);
    TWXI_LAUNCH_CHECK();
    return TWXI_OK;
}

__global__ void split3_kernel(size_t n, const double* src, const int32_t* status, int per_point, double* a, double* b, double* c) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const bool good = status[i / per_point] == TWXI_ST_OK;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    a[i] = good ? src[3 * i] : nan;
    b[i] = good ? src[3 * i + 1] : nan;
    c[i] = good ? src[3 * i + 2] : nan;
}
int launch_split3(cudaStream_t s, size_t n, const double* src, const int32_t* status, int per_point, double* a, double* b,
                  double* c) {
    if (n == 0) return TWXI_OK;
    split3_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(n, src, status, per_point, a, b, c);
    TWXI_LAUNCH_CHECK();
    return TWXI_OK;
}

}  // namespace twxi

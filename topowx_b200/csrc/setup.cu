// Stage a4-a5: per-point smoothed neighbour counts and variogram parameters for all 12 months
// (replaces KrigTair.__get_nnghs / GwrTairAnom.__get_nnghs / KrigTair.__get_vario_params,
// twx/interp/interp_tair.py:821-851 and :245-259), plus the point->candidate WGS-84 distances the
// kriging stage needs for c0 (gstat uses great-circle distances for long/lat data, interp.R:218-221).
// One warp per point; everything is a handful of warp reductions over <= 255 candidates.
#include "twxi_internal.cuh"

namespace twxi {

constexpr int SETUP_THREADS = 128;
// the GWR fits an intercept and the five GWR_TREND_VARS (interp_tair.py:47): with fewer neighbours X'WX is singular
constexpr int GWR_MIN_NNGHS = 1 + 5;
// the kriging trend is an intercept and four drift columns (lon, lat, elev, lst; interp.R:256): with fewer neighbours
// G = X'V^-1X is singular in exact arithmetic, and a rounded pivot must not decide it
constexpr int KED_MIN_NNGHS = 1 + 4;

struct SetupArgs {
    StnTable st;
    int npts, k1;
    const double* qlat;
    const double* qlon;
    const int32_t* idx;
    const double* dist;
    const int32_t* norm_override;   // [npts] or null: krig(nnghs=...) for month override_mth
    const int32_t* anom_override;   // [npts] or null
    int only_mth;                   // 0 = all months, else the single month (1..12) that is needed
    int need_norm, need_anom, need_vario;
    int32_t* nn;
    double* vario;
    double* h0;
    int32_t* status;
};

__device__ __forceinline__ double bisquare(double d, double dbw) {   // station_select.py:169
    double r = d / dbw;
    double u = __dsub_rn(1.0, __dmul_rn(r, r));
    return __dmul_rn(u, u);
}

__global__ void __launch_bounds__(SETUP_THREADS) nngh_params_kernel(SetupArgs a) {
    const int q = blockIdx.x * (SETUP_THREADS / 32) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (q >= a.npts) return;
    if (a.status[q] != TWXI_ST_OK) return;
    const int n = a.st.n, k1 = a.k1;
    const int32_t* idx = a.idx + (size_t)q * k1;
    const double* dist = a.dist + (size_t)q * k1;
    int st = TWXI_ST_OK;

    // weights of the DFLT_INIT_NNGHS = 100 nearest (interp_tair.py:823, 247); bandwidth = 101st distance
    const int ninit = TWXI_INIT_NNGHS;
    int knorm[12], kanom[12];
    const bool need_smooth = (a.need_norm && !a.norm_override) || (a.need_anom && !a.anom_override);
    if (!need_smooth) {
        for (int m = 0; m < 12; ++m) {
            const bool need_m = a.only_mth == 0 || a.only_mth == m + 1;
            knorm[m] = (need_m && a.need_norm) ? a.norm_override[q] : 0;
            kanom[m] = (need_m && a.need_anom) ? a.anom_override[q] : 0;
        }
    } else if (k1 <= ninit) {
        st = TWXI_ST_TOO_FEW_STNS;                             // IndexError: set_ngh_stns(100) with < 101 stations
    } else {
        // lane L < 24 owns one (kind, month) column of the station-major table: L = month for optim_nnghs, 12 + month for
        // optim_nnghs_anom.  Per neighbour the warp reads ONE 192-byte run; weights and indices are staged per warp.
        __shared__ double s_w[SETUP_THREADS / 32][TWXI_INIT_NNGHS];
        __shared__ int s_s[SETUP_THREADS / 32][TWXI_INIT_NNGHS];
        const int wq = threadIdx.x >> 5;
        const double dbw = dist[ninit];
        for (int j = lane; j < ninit; j += 32) {
            s_w[wq][j] = bisquare(dist[j], dbw);
            s_s[wq][j] = idx[j];
        }
        __syncwarp();
        double num = 0.0, den = 0.0;
        if (lane < 24) {
            const double* col = a.st.optim2 + lane;
#pragma unroll 4
            for (int j = 0; j < ninit; ++j) {
                const double v = col[(size_t)s_s[wq][j] * 24];
                const double w = s_w[wq][j];
                if (isfinite(v)) { num += v * w; den += w; }
            }
        }
        // finite-count is implied by den > 0 unless every finite neighbour has weight 0 (ZeroDivisionError in np.average ->
        // same per-point failure); np.round: half to even
        const int kmine = den > 0 ? (int)rint(num / den) : -1;
        for (int m = 0; m < 12; ++m) {
            int kn = __shfl_sync(0xffffffffu, kmine, m), ka = __shfl_sync(0xffffffffu, kmine, 12 + m);
            if (a.norm_override) kn = a.norm_override[q];
            if (a.anom_override) ka = a.anom_override[q];
            const bool need_m = a.only_mth == 0 || a.only_mth == m + 1;
            knorm[m] = (need_m && a.need_norm) ? kn : 0;      // 0 = month / kind not requested
            kanom[m] = (need_m && a.need_anom) ? ka : 0;
        }
    }
    int kmax = 0;
    if (st == TWXI_ST_OK) {
        for (int m = 0; m < 12; ++m) {
            const bool need_m = a.only_mth == 0 || a.only_mth == m + 1;
            if (!need_m) continue;
            if ((a.need_norm && knorm[m] < 0) || (a.need_anom && kanom[m] < 0)) { st = TWXI_ST_NO_NNGHS; break; }
            if (knorm[m] >= k1 || kanom[m] >= k1) { st = TWXI_ST_TOO_FEW_STNS; break; }
            if ((a.need_norm && knorm[m] < KED_MIN_NNGHS) || (a.need_anom && kanom[m] < GWR_MIN_NNGHS)) {
                st = TWXI_ST_SINGULAR;
                break;
            }
            kmax = max(kmax, knorm[m]);
        }
    }
    if (st == TWXI_ST_OK) {
        // smoothed variogram parameters over the k_norm neighbours (interp_tair.py:837-851)
        for (int m = 0; m < 12; ++m) {
            const int k = knorm[m];
            if (k < 1 || !a.need_vario) continue;
            const double dbw = dist[k];
            double sw = 0, snug = 0, sps = 0, srg = 0;
            for (int j = lane; j < k; j += 32) {
                const double* v = a.st.vario2 + (size_t)idx[j] * 36 + m * 3;    // (nug, psill, rng): one 24-byte run
                const double vn = v[0];
                if (isfinite(vn)) {
                    double w = bisquare(dist[j], dbw);
                    sw += w;
                    snug += vn * w;
                    sps += v[1] * w;
                    srg += v[2] * w;
                }
            }
            sw = warp_sum(sw); snug = warp_sum(snug); sps = warp_sum(sps); srg = warp_sum(srg);
            if (!(sw > 0)) { st = TWXI_ST_NO_VARIO; break; }
            if (lane == 0) {
                double* v = a.vario + ((size_t)q * 12 + m) * 3;
                v[0] = snug / sw; v[1] = sps / sw; v[2] = srg / sw;
            }
        }
    }
    if (st == TWXI_ST_OK) {
        const double qlat = a.qlat[q], qlon = a.qlon[q];
        for (int j = lane; j < kmax; j += 32) {
            int s = idx[j];
            a.h0[(size_t)q * k1 + j] = gcdist_sp(qlon, qlat, a.st.lon[s], a.st.lat[s]);
        }
        if (lane < 12) {
            a.nn[(size_t)q * 24 + lane] = knorm[lane];
            a.nn[(size_t)q * 24 + 12 + lane] = kanom[lane];
        }
    }
    if (lane == 0 && st != TWXI_ST_OK) a.status[q] = st;
}

int launch_nngh_params(Ctx& c, Batch& b, const int32_t* norm_override, const int32_t* anom_override, int only_mth,
                       int need_norm, int need_anom, int need_vario) {
    if (b.npts <= 0) return TWXI_OK;
    SetupArgs a;
    a.st = c.st; a.npts = b.npts; a.k1 = b.k1; a.qlat = b.lat; a.qlon = b.lon; a.idx = b.idx; a.dist = b.dist;
    a.norm_override = norm_override; a.anom_override = anom_override; a.only_mth = only_mth;
    a.need_norm = need_norm; a.need_anom = need_anom; a.need_vario = need_vario;
    a.nn = b.nn; a.vario = b.vario; a.h0 = b.h0; a.status = b.status;
    int per = SETUP_THREADS / 32;
    nngh_params_kernel<<<(b.npts + per - 1) / per, SETUP_THREADS, 0, c.stream>>>(a);
    TWXI_LAUNCH_CHECK();
    return TWXI_OK;
}

}  // namespace twxi

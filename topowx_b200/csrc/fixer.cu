// Stages around the per-variable kernels:
//  * unpack_chunk  – step25's per-cell copy of the work-chunk planes into the point record
//                    (scripts/step25_mpi_interp_tair.py:132-144, plane layout twx/interp/tiling.py:205-213) and the
//                    climate-division lookup that raises KeyError in PtInterpTair.interp_pt (interp_tair.py:563,572);
//  * fixer         – tmin_tmax_fixer (interp_tair.py:143-197), the 1981-2010 normals recomputation after a fix
//                    (:583-590), std_err (:816) and the output quantisation of step25:163-172;
//  * finalize      – per-variable outputs of InterpTair.interp (:396-439).
// One warp per cell; lanes run over days.
#include "twxi_internal.cuh"

namespace twxi {

__device__ __forceinline__ bool in_set(const double* set, int n, double v) {
    if (n < 0) return true;                                   // no check requested
    for (int i = 0; i < n; ++i)
        if (set[i] == v) return true;                         // NaN never matches (dict lookup of nan -> KeyError)
    return false;
}

__global__ void unpack_chunk_kernel(const double* __restrict__ wrk, int ncell, const double* cd_a, int n_a,
                                    const double* cd_b, int n_b, Batch bmin, Batch bmax) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= ncell) return;
    const size_t P = (size_t)ncell;
    const double mask = wrk[2 * P + q];
    const double lat = wrk[3 * P + q], lon = wrk[4 * P + q], elev = wrk[5 * P + q], tdi = wrk[6 * P + q];
    bmin.lat[q] = lat; bmin.lon[q] = lon; bmin.elev[q] = elev; bmin.tdi[q] = tdi;
    bmax.lat[q] = lat; bmax.lon[q] = lon; bmax.elev[q] = elev; bmax.tdi[q] = tdi;
#pragma unroll
    for (int m = 0; m < 12; ++m) {
        bmin.lst[(size_t)q * 12 + m] = wrk[(size_t)(8 + m) * P + q];      // "tminMM" = LST night
        bmax.lst[(size_t)q * 12 + m] = wrk[(size_t)(20 + m) * P + q];     // "tmaxMM" = LST day
    }
    int sa = TWXI_ST_OK, sb = TWXI_ST_OK;
    if (mask == 0.0) {                                        // `if wrk_chk[2, r, c]:` (NaN is truthy)
        sa = sb = TWXI_ST_MASKED;
    } else {
        const double cd = wrk[7 * P + q];
        if (!in_set(cd_a, n_a, cd)) sa = TWXI_ST_CLIMDIV;
        if (!in_set(cd_b, n_b, cd)) sb = TWXI_ST_CLIMDIV;
    }
    bmin.status[q] = sa;
    bmax.status[q] = sb;
}

int launch_unpack_chunk(cudaStream_t s, const double* wrk, int ny, int nx, const double* cd_a, int n_a,
                        const double* cd_b, int n_b, Batch& bmin, Batch& bmax) {
    const int ncell = ny * nx;
    unpack_chunk_kernel<<<(ncell + 255) / 256, 256, 0, s>>>(wrk, ncell, cd_a, n_a, cd_b, n_b, bmin, bmax);
    TWXI_LAUNCH_CHECK();
    return TWXI_OK;
}

__global__ void cells_status_kernel(int ncell, const double* climdiv, const double* cd_a, int n_a,
                                    const double* cd_b, int n_b, int32_t* sa, int32_t* sb) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= ncell) return;
    int a = TWXI_ST_OK, b = TWXI_ST_OK;
    if (climdiv) {
        if (!in_set(cd_a, n_a, climdiv[q])) a = TWXI_ST_CLIMDIV;
        if (!in_set(cd_b, n_b, climdiv[q])) b = TWXI_ST_CLIMDIV;
    }
    sa[q] = a;
    sb[q] = b;
}

int launch_cells_status(cudaStream_t s, int ncell, const double* climdiv, const double* cd_a, int n_a,
                        const double* cd_b, int n_b, int32_t* sa, int32_t* sb) {
    cells_status_kernel<<<(ncell + 255) / 256, 256, 0, s>>>(ncell, climdiv, cd_a, n_a, cd_b, n_b, sa, sb);
    TWXI_LAUNCH_CHECK();
    return TWXI_OK;
}

struct FixerArgs {
    int ncell, ndays, fix_invalid;
    ObsTable ob;
    double* dmin;               // [ncell][ndays] daily (modified in place by fixes), may be null (normals only)
    double* dmax;
    const double *mean_min, *var_min, *mean_max, *var_max;    // [ncell][12]
    const int32_t *st_min, *st_max;
    // outputs
    uint8_t* status;
    double *nmin, *nmax, *semin, *semax;                      // f8 [ncell][12]
    int16_t *qmin, *qmax;                                     // i16 [ndays][ncell]
    float *fnmin, *fnmax, *fsemin, *fsemax;                   // f4 [12][ncell]
    int32_t* ninvalid;
};

__global__ void __launch_bounds__(128) fixer_kernel(FixerArgs a) {
    const int q = blockIdx.x * 4 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (q >= a.ncell) return;
    const int nd = a.ndays;
    const size_t P = (size_t)a.ncell;
    int st = a.st_min[q];
    if (st == TWXI_ST_OK) st = a.st_max[q];
    double* tmin = a.dmin ? a.dmin + (size_t)q * nd : nullptr;
    double* tmax = a.dmax ? a.dmax + (size_t)q * nd : nullptr;
    int ninv = 0;
    double nrm_min[12], nrm_max[12];                          // lane m (<12) keeps month m in [0]; simple arrays
    bool recompute = false;

    if (st == TWXI_ST_OK && tmin && a.fix_invalid) {
        // invalid_days = nonzero(tmin >= tmax) on the unfixed series (interp_tair.py:171)
        ninv = fix_inverted(tmin, tmax, 0, 0, nd, nd, lane, st);
        recompute = st == TWXI_ST_OK && ninv > 0;
    }

    if (st == TWXI_ST_OK) {
#pragma unroll
        for (int m = 0; m < 12; ++m) {
            nrm_min[m] = a.mean_min[(size_t)q * 12 + m];
            nrm_max[m] = a.mean_max[(size_t)q * 12 + m];
        }
        if (recompute) {
            // mean over years of the monthly means of the 1981-2010 days (interp_tair.py:583-590)
            const int nyr = a.ob.ngroups / 12;
            for (int m = 0; m < 12; ++m) {
                double accmin = 0.0, accmax = 0.0;
                for (int y = 0; y < nyr; ++y) {
                    const int g = y * 12 + m;
                    const int s0 = a.ob.grp_start[g], len = a.ob.grp_len[g];
                    double smin = 0.0, smax = 0.0;
                    group_lane_days(0, len, lane, [&](int o) { smin += tmin[s0 + o]; smax += tmax[s0 + o]; });
                    smin = warp_sum(smin); smax = warp_sum(smax);
                    accmin += smin / len;                     // len == 0 -> NaN, like np.mean of an empty slice
                    accmax += smax / len;
                }
                nrm_min[m] = accmin / nyr;
                nrm_max[m] = accmax / nyr;
            }
        }
    }

    // ---- outputs (every cell writes either results or fill values) -----------------------------------------
    const bool good = st == TWXI_ST_OK;
    if (lane == 0) {
        a.status[q] = (uint8_t)st;
        if (a.ninvalid) a.ninvalid[q] = good ? ninv : TWXI_FILL_I4;
    }
#pragma unroll
    for (int m = 0; m < 12; ++m) {
        if (lane == m) {
            double vmin = 0, vmax = 0, se_min = 0, se_max = 0;
            if (good) {
                vmin = a.var_min[(size_t)q * 12 + m];
                vmax = a.var_max[(size_t)q * 12 + m];
                se_min = vmin >= 0 ? sqrt(vmin) : 0.0;        // interp_tair.py:816
                se_max = vmax >= 0 ? sqrt(vmax) : 0.0;
            }
            if (a.nmin) {
                a.nmin[(size_t)q * 12 + m] = good ? nrm_min[m] : TWXI_FILL_F8;
                a.nmax[(size_t)q * 12 + m] = good ? nrm_max[m] : TWXI_FILL_F8;
                a.semin[(size_t)q * 12 + m] = good ? se_min : TWXI_FILL_F8;
                a.semax[(size_t)q * 12 + m] = good ? se_max : TWXI_FILL_F8;
            }
            if (a.fnmin) {
                a.fnmin[(size_t)m * P + q] = good ? (float)nrm_min[m] : TWXI_FILL_F4;
                a.fnmax[(size_t)m * P + q] = good ? (float)nrm_max[m] : TWXI_FILL_F4;
                a.fsemin[(size_t)m * P + q] = good ? (float)se_min : TWXI_FILL_F4;
                a.fsemax[(size_t)m * P + q] = good ? (float)se_max : TWXI_FILL_F4;
            }
        }
    }
    if (a.qmin) {
        for (int d = lane; d < nd; d += 32) {
            a.qmin[(size_t)d * P + q] = good ? quantize(tmin[d]) : TWXI_FILL_I2;
            a.qmax[(size_t)d * P + q] = good ? quantize(tmax[d]) : TWXI_FILL_I2;
        }
    } else if (!good && tmin) {
        for (int d = lane; d < nd; d += 32) { tmin[d] = TWXI_FILL_F8; tmax[d] = TWXI_FILL_F8; }
    }
}

int launch_fixer(Ctx& cmin, Ctx& cmax, int ncells, int fix_invalid, int have_daily, const ChunkOut& out, double* f8) {
    if (ncells <= 0) return TWXI_OK;
    const size_t n12 = (size_t)ncells * 12;
    FixerArgs a;
    a.ncell = ncells; a.ndays = cmin.ob.ndays; a.fix_invalid = fix_invalid; a.ob = cmin.ob;
    a.dmin = have_daily ? cmin.b.daily : nullptr;
    a.dmax = have_daily ? cmax.b.daily : nullptr;
    a.mean_min = cmin.b.mean; a.var_min = cmin.b.var; a.mean_max = cmax.b.mean; a.var_max = cmax.b.var;
    a.st_min = cmin.b.status; a.st_max = cmax.b.status;
    a.status = out.st;
    a.nmin = f8; a.nmax = f8 ? f8 + n12 : nullptr; a.semin = f8 ? f8 + 2 * n12 : nullptr; a.semax = f8 ? f8 + 3 * n12 : nullptr;
    a.qmin = have_daily ? out.q[0] : nullptr; a.qmax = have_daily ? out.q[1] : nullptr;
    a.fnmin = out.norm[0]; a.fnmax = out.norm[1]; a.fsemin = out.se[0]; a.fsemax = out.se[1]; a.ninvalid = out.ninv;
    fixer_kernel<<<(ncells + 3) / 4, 128, 0, cmin.stream>>>(a);
    TWXI_LAUNCH_CHECK();
    return TWXI_OK;
}

// ---- single-variable finalisation (InterpTair.interp outputs) ----------------------------------------------
__global__ void finalize_points_kernel(int npts, int ndays, const int32_t* st, const double* mean, const double* var,
                                       double* daily, double* norms, double* se, double* var_out, uint8_t* status) {
    const int q = blockIdx.x * 4 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (q >= npts) return;
    const bool good = st[q] == TWXI_ST_OK;
    if (lane == 0 && status) status[q] = (uint8_t)st[q];
    if (lane < 12) {
        const size_t o = (size_t)q * 12 + lane;
        const double v = good ? var[o] : TWXI_FILL_F8;
        if (norms) norms[o] = good ? mean[o] : TWXI_FILL_F8;
        if (se) se[o] = good ? (v >= 0 ? sqrt(v) : 0.0) : TWXI_FILL_F8;
        if (var_out) var_out[o] = v;
    }
    if (daily && !good)
        for (int d = lane; d < ndays; d += 32) daily[(size_t)q * ndays + d] = TWXI_FILL_F8;
}

int launch_finalize_points(Ctx& c, Batch& b, double* daily, double* norms, double* se, double* var_out,
                           uint8_t* status) {
    if (b.npts <= 0) return TWXI_OK;
    finalize_points_kernel<<<(b.npts + 3) / 4, 128, 0, c.stream>>>(b.npts, c.ob.ndays, b.status, b.mean, b.var, daily,
                                                                  norms, se, var_out, status);
    TWXI_LAUNCH_CHECK();
    return TWXI_OK;
}

__global__ void status_to_u8_kernel(int n, const int32_t* in, uint8_t* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (uint8_t)in[i];
}
int launch_status_to_u8(cudaStream_t s, int n, const int32_t* in, uint8_t* out) {
    if (n <= 0) return TWXI_OK;
    status_to_u8_kernel<<<(n + 255) / 256, 256, 0, s>>>(n, in, out);
    TWXI_LAUNCH_CHECK();
    return TWXI_OK;
}

// masked 12-column copies for the stage entry points (krig single month etc.)
__global__ void gather_month_kernel(int npts, int mth0, const int32_t* st, const double* src12, double* dst,
                                    int dst_stride) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= npts) return;
    const bool good = st[q] == TWXI_ST_OK;
    if (mth0 >= 0) dst[q] = good ? src12[(size_t)q * 12 + mth0] : TWXI_FILL_F8;
    else
        for (int m = 0; m < 12; ++m) dst[(size_t)q * dst_stride + m] = good ? src12[(size_t)q * 12 + m] : TWXI_FILL_F8;
}
int launch_gather_month(cudaStream_t s, int npts, int mth0, const int32_t* st, const double* src12, double* dst) {
    if (npts <= 0) return TWXI_OK;
    gather_month_kernel<<<(npts + 255) / 256, 256, 0, s>>>(npts, mth0, st, src12, dst, 12);
    TWXI_LAUNCH_CHECK();
    return TWXI_OK;
}

// variogram parameters [npts][12][3] -> [npts][12|1][3], NaN for failed points / months without a system
__global__ void gather_vario_kernel(int npts, int mth0, const int32_t* st, const int32_t* nn, const double* src, double* dst) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int nm = mth0 >= 0 ? 1 : 12;
    if (i >= npts * nm) return;
    const int q = i / nm, m = mth0 >= 0 ? mth0 : i % nm;
    const bool good = st[q] == TWXI_ST_OK && nn[(size_t)q * 24 + m] > 0;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    for (int k = 0; k < 3; ++k) dst[(size_t)i * 3 + k] = good ? src[((size_t)q * 12 + m) * 3 + k] : nan;
}
int launch_gather_vario(cudaStream_t s, int npts, int mth0, const int32_t* st, const int32_t* nn, const double* src,
                        double* dst) {
    if (npts <= 0) return TWXI_OK;
    const int n = npts * (mth0 >= 0 ? 1 : 12);
    gather_vario_kernel<<<(n + 255) / 256, 256, 0, s>>>(npts, mth0, st, nn, src, dst);
    TWXI_LAUNCH_CHECK();
    return TWXI_OK;
}

}  // namespace twxi

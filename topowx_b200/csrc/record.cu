// Day windows of a work chunk's record (twxi_tile_begin / twxi_tile_days / twxi_tile_end).
//
// twxi_interp_chunk holds a chunk's whole daily record on the device (f64 [ncell][ndays] per variable: 12.4 GB for a
// 250 x 250 tile over 1948-2015).  Here the day-independent work (kNN, neighbour counts, kriging, GWR hat rows) runs once
// at begin and the record is emitted in consecutive windows of any length; each window costs the GWR daily apply, the
// Tmin >= Tmax fixer and the quantisation only.  The windows concatenate to exactly the bytes of twxi_interp_chunk, because
// each step calls the helper its whole-record kernel calls (twxi_internal.cuh):
//  * apply  - hat_dot with the stored hat rows, as gwr_kernel's day loop;
//  * fixer  - fix_inverted over carry (the last 15 fixed days) + window + 15 unfixed look-ahead days, as fixer_kernel over
//             the record: the fix of day x reads fixed days x-15..x-1 and unfixed days x..x+15, wherever the window
//             boundaries are;
//  * normals- group_lane_days over the window's part of each 1981-2010 (year, month) group, then warp_sum and the running
//             sum over years as in fixer_kernel, with the lane partials of an unfinished group carried over.
// A fixed day is valid (tavg -/+ half, half > 0), so only the fix of day 0 can find no valid day in its window; that
// decision falls in the first window, which always computes days 1..15 as look-ahead.
//
// twxi_tile_days_mth adds the monthly means of the emitted int16 counts (tile_month_kernel, after tile_fix_kernel):
// exact int32 sums per (cell, month run), so no order or window boundary can change them, with the sum of the run that
// the window leaves open carried to the next window.
#include "twxi_internal.cuh"

namespace twxi {

constexpr int TAIL = 15;                     // half-window of the fixer (interp_tair.py:177-183)
constexpr int REC_THREADS = 256;
constexpr int REC_WARPS = REC_THREADS / 32;
constexpr int REC_MAXK = 256;

__global__ void tile_init_kernel(int ncell, const int32_t* st_min, const int32_t* st_max, int32_t* status,
                                 int32_t* ninv, double* carry, double* gpart, double* gacc) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= ncell) return;
    int st = st_min[q];
    if (st == TWXI_ST_OK) st = st_max[q];
    status[q] = st;
    ninv[q] = 0;
    for (int v = 0; v < 2; ++v) {
        for (int i = 0; i < TAIL; ++i) carry[((size_t)v * ncell + q) * TAIL + i] = 0.0;
        for (int i = 0; i < 32; ++i) gpart[((size_t)v * ncell + q) * 32 + i] = 0.0;
        for (int i = 0; i < 12; ++i) gacc[((size_t)v * ncell + q) * 12 + i] = 0.0;
    }
}

int launch_tile_init(cudaStream_t s, TileState& t, const Batch& bmin, const Batch& bmax) {
    const size_t n12 = (size_t)t.ncell * 12 * 8;
    TWXI_CUDA(cudaMemcpyAsync(t.mean, bmin.mean, n12, cudaMemcpyDeviceToDevice, s));
    TWXI_CUDA(cudaMemcpyAsync(t.mean + (size_t)t.ncell * 12, bmax.mean, n12, cudaMemcpyDeviceToDevice, s));
    TWXI_CUDA(cudaMemcpyAsync(t.var, bmin.var, n12, cudaMemcpyDeviceToDevice, s));
    TWXI_CUDA(cudaMemcpyAsync(t.var + (size_t)t.ncell * 12, bmax.var, n12, cudaMemcpyDeviceToDevice, s));
    tile_init_kernel<<<(t.ncell + 255) / 256, 256, 0, s>>>(t.ncell, bmin.status, bmax.status, t.status, t.ninv, t.carry,
                                                          t.gpart, t.gacc);
    TWXI_LAUNCH_CHECK();
    return TWXI_OK;
}

struct ApplyArgs {
    int ncell, kh, nd, w0, wst;
    const float* obsT;
    const int* day_of_pos;
    const int32_t* status;
    const int32_t* hk;
    const int32_t* hidx;
    const double* hz;
    const double* hoff;
    double* out;               // [ncell][wst]: day w0 + i at column TAIL + i
    int p0[12], cnt[12];
};

// Items are (cell, month), month-major like gwr_kernel; lanes are the days of the month inside window + look-ahead, which
// are one contiguous run of month-major positions, so every neighbour is a coalesced 128-byte gather of obsT.
__global__ void __launch_bounds__(REC_THREADS, 4) tile_apply_kernel(ApplyArgs a) {
    __shared__ __align__(16) double s_z[REC_WARPS][REC_MAXK];
    __shared__ __align__(16) int s_off[REC_WARPS][REC_MAXK];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long item = (long long)blockIdx.x * REC_WARPS + warp;
    if (item >= (long long)a.ncell * 12) return;
    const int q = (int)(item % a.ncell);
    const int m = (int)(item / a.ncell);
    const int D = a.cnt[m];
    if (D == 0 || a.status[q] != TWXI_ST_OK) return;
    const size_t qm = (size_t)q * 12 + m;
    const int k = a.hk[qm];
    const int32_t* hidx = a.hidx + qm * a.kh;
    const double* hz = a.hz + qm * a.kh;
    const int kpad = (k + 3) & ~3;                            // the 4- and 8-wide passes read int4 / double2 rows
    for (int j = lane; j < kpad; j += 32) {
        s_z[warp][j] = j < k ? hz[j] : 0.0;
        s_off[warp][j] = j < k ? hidx[j] * a.nd : 0;
    }
    __syncwarp();
    const double off = a.hoff[qm];
    const int p0 = a.p0[m];
    double* out = a.out + (size_t)q * a.wst + TAIL - a.w0;
    for (int d0 = 0; d0 < D; d0 += 32) {
        const int d = d0 + lane;
        const bool valid = d < D;
        const double v = hat_dot(a.obsT + p0 + (valid ? d : 0), s_z[warp], s_off[warp], k) + off;
        if (valid) out[a.day_of_pos[p0 + d]] = v;
    }
}

struct FixArgs {
    int ncell, nd, w0, nwin, la, wst;
    double* dmin;              // [ncell][wst] window dailies of tmin / tmax (fixed in place)
    double* dmax;
    int32_t* status;
    int32_t* ninv;
    double* carry;             // [2][ncell][TAIL]
    double* gpart;             // [2][ncell][32]
    double* gacc;              // [2][ncell][12]
    const int* grp_start;
    const int* grp_len;
    int g0, g1;
    int16_t* qmin;             // [nwin][ncell]
    int16_t* qmax;
};

// The part of group g inside the window (group_lane_days, as fixer_kernel sums whole groups); the group's mean joins the
// running sum over years once its last day has been seen.
__device__ __forceinline__ void group_part(const FixArgs& a, int g, int lane, const double* buf, double& part,
                                           double* acc) {
    const int gs = a.grp_start[g], len = a.grp_len[g];
    const int lo = max(gs, a.w0) - gs, hi = min(gs + len, a.w0 + a.nwin) - gs;
    group_lane_days(lo, hi, lane, [&](int o) { part += buf[gs + o - a.w0 + TAIL]; });
    if (gs + len <= a.w0 + a.nwin) {
        const double s = warp_sum(part);
        *acc += s / len;
        part = 0.0;
    }
}

__global__ void __launch_bounds__(128) tile_fix_kernel(FixArgs a) {
    const int q = blockIdx.x * 4 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (q >= a.ncell) return;
    const size_t P = (size_t)a.ncell;
    int st = a.status[q];
    double* tmin = a.dmin + (size_t)q * a.wst;                // column c holds day w0 - TAIL + c
    double* tmax = a.dmax + (size_t)q * a.wst;
    double* cmin = a.carry + (size_t)q * TAIL;
    double* cmax = a.carry + (P + q) * TAIL;
    int ninv = 0;
    if (st == TWXI_ST_OK) {
        if (lane < TAIL) { tmin[lane] = cmin[lane]; tmax[lane] = cmax[lane]; }
        __syncwarp();
        // the window's days are columns TAIL .. TAIL + nwin - 1; columns up to nwin + TAIL + la - 1 are computed
        ninv = fix_inverted(tmin, tmax, a.w0 - TAIL, TAIL, a.nwin, a.nwin + TAIL + a.la, lane, st);
    }
    const bool good = st == TWXI_ST_OK;
    if (good) {
        for (int v = 0; v < 2; ++v) {
            const double* buf = v ? tmax : tmin;
            double* acc = a.gacc + (v * P + q) * 12;
            double part = a.gpart[(v * P + q) * 32 + lane];
            for (int g = a.g0; g < a.g1; ++g)
                if (a.grp_len[g] > 0) group_part(a, g, lane, buf, part, acc + g % 12);   // empty groups: NaN at the end
            a.gpart[(v * P + q) * 32 + lane] = part;
        }
        // carry: fixed days w0 + nwin - 15 .. w0 + nwin - 1 = columns nwin .. nwin + 14
        double c0 = 0.0, c1 = 0.0;
        if (lane < TAIL) { c0 = tmin[a.nwin + lane]; c1 = tmax[a.nwin + lane]; }
        __syncwarp();
        if (lane < TAIL) { cmin[lane] = c0; cmax[lane] = c1; }
    }
    if (lane == 0) {
        a.status[q] = st;
        a.ninv[q] += ninv;
    }
    for (int d = lane; d < a.nwin; d += 32) {
        a.qmin[(size_t)d * P + q] = good ? quantize(tmin[TAIL + d]) : TWXI_FILL_I2;
        a.qmax[(size_t)d * P + q] = good ? quantize(tmax[TAIL + d]) : TWXI_FILL_I2;
    }
}

int launch_tile_apply(cudaStream_t s, TileState& t, const Ctx& cmin, const Ctx& cmax, const WindowSpan& w) {
    const int wst = w.nwin + 2 * TAIL;
    void* p;
    const int rc = t.win.get(&p, (size_t)2 * t.ncell * wst * 8);
    if (rc != TWXI_OK) return rc;
    double* buf = static_cast<double*>(p);
    const Ctx* cs[2] = {&cmin, &cmax};
    for (int v = 0; v < 2; ++v) {
        ApplyArgs a;
        a.ncell = t.ncell; a.kh = t.kh; a.nd = cs[v]->ob.ndays; a.w0 = w.w0; a.wst = wst;
        a.obsT = cs[v]->ob.obsT; a.day_of_pos = cs[v]->ob.day_of_pos; a.status = t.status;
        const size_t n12 = (size_t)v * t.ncell * 12;
        a.hk = t.hk + n12; a.hidx = t.hidx + n12 * t.kh; a.hz = t.hz + n12 * t.kh; a.hoff = t.hoff + n12;
        a.out = buf + (size_t)v * t.ncell * wst;
        for (int m = 0; m < 12; ++m) { a.p0[m] = w.p0[v][m]; a.cnt[m] = w.cnt[v][m]; }
        const long long items = (long long)t.ncell * 12;
        tile_apply_kernel<<<(unsigned)((items + REC_WARPS - 1) / REC_WARPS), REC_THREADS, 0, s>>>(a);
        TWXI_LAUNCH_CHECK();
    }
    return TWXI_OK;
}

int launch_tile_fix(cudaStream_t s, TileState& t, const Ctx& cmin, const WindowSpan& w, int16_t* qmin, int16_t* qmax) {
    const int wst = w.nwin + 2 * TAIL;
    double* buf = static_cast<double*>(t.win.p);              // the window dailies of launch_tile_apply
    FixArgs f;
    f.ncell = t.ncell; f.nd = t.ndays; f.w0 = w.w0; f.nwin = w.nwin; f.la = w.la; f.wst = wst;
    f.dmin = buf; f.dmax = buf + (size_t)t.ncell * wst;
    f.status = t.status; f.ninv = t.ninv; f.carry = t.carry; f.gpart = t.gpart; f.gacc = t.gacc;
    f.grp_start = cmin.ob.grp_start; f.grp_len = cmin.ob.grp_len; f.g0 = w.g0; f.g1 = w.g1;
    f.qmin = qmin; f.qmax = qmax;
    tile_fix_kernel<<<(t.ncell + 3) / 4, 128, 0, s>>>(f);
    TWXI_LAUNCH_CHECK();
    return TWXI_OK;
}

struct MonthArgs {
    int ncell, w0, w1, g0, g1;
    const int* run_start;      // month runs of the record (Ctx::mrun_*)
    const int* run_len;
    const int32_t* status;
    int32_t* carry;            // [2][ncell]
    const int16_t* qmin;       // [w1 - w0][ncell] the window's quantised tmin / tmax
    const int16_t* qmax;
    float* fmin;               // [nmth][ncell] monthly means of tmin / tmax
    float* fmax;
};

// One thread per (cell, variable), days in order: every day is one coalesced [d][ncell] row.  S / n * 0.01f in double,
// rounded once to float (no contraction).  Cells that are not ok (masked, failed at begin or by the fixer of the first
// window, which ran before this kernel) have fill counts and get fill in every month.
__global__ void tile_month_kernel(MonthArgs a) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= a.ncell) return;
    const int v = blockIdx.y;
    const size_t P = (size_t)a.ncell;
    const int16_t* in = (v ? a.qmax : a.qmin) + q;
    float* out = (v ? a.fmax : a.fmin) + q;
    const bool good = a.status[q] == TWXI_ST_OK;
    int s = a.w0 == 0 ? 0 : a.carry[v * P + q];               // the first window starts every sum at zero
    int d = a.w0;
    for (int g = a.g0; g < a.g1; ++g) {
        const int gend = a.run_start[g] + a.run_len[g];
        const int end = min(gend, a.w1);
        if (good) {
#pragma unroll 8
            for (; d < end; ++d) s += in[(size_t)(d - a.w0) * P];
        }
        d = end;
        if (gend <= a.w1) {
            const double mean = __dmul_rn(__ddiv_rn((double)s, (double)a.run_len[g]), (double)0.01f);
            out[(size_t)(g - a.g0) * P] = good ? (float)mean : TWXI_FILL_F4;
            s = 0;
        }
    }
    a.carry[v * P + q] = s;
}

int launch_tile_month(cudaStream_t s, TileState& t, const Ctx& cmin, const WindowSpan& w, const MonthSpan& m,
                      const int16_t* qmin, const int16_t* qmax, float* fmin, float* fmax) {
    MonthArgs a;
    a.ncell = t.ncell; a.w0 = w.w0; a.w1 = w.w0 + w.nwin; a.g0 = m.g0; a.g1 = m.g1;
    a.run_start = cmin.mrun_start; a.run_len = cmin.mrun_len;
    a.status = t.status; a.carry = t.mcarry;
    a.qmin = qmin; a.qmax = qmax; a.fmin = fmin; a.fmax = fmax;
    tile_month_kernel<<<dim3((t.ncell + 255) / 256, 2), 256, 0, s>>>(a);
    TWXI_LAUNCH_CHECK();
    return TWXI_OK;
}

__global__ void tile_end_kernel(int ncell, int ngroups, const int* grp_len, const int32_t* status, const int32_t* ninv,
                                const double* mean, const double* var, const double* gacc, float* fnmin, float* fnmax,
                                float* fsemin, float* fsemax, int32_t* ninvalid, uint8_t* st_out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ncell * 12) return;
    const int q = i / 12, m = i % 12;
    const size_t P = (size_t)ncell;
    const int st = status[q];
    const bool good = st == TWXI_ST_OK;
    if (m == 0) {
        st_out[q] = (uint8_t)st;
        ninvalid[q] = good ? ninv[q] : TWXI_FILL_I4;
    }
    const bool recompute = good && ninv[q] > 0;
    float* fn[2] = {fnmin, fnmax};
    float* fs[2] = {fsemin, fsemax};
    for (int v = 0; v < 2; ++v) {
        const size_t o = (v * P + q) * 12 + m;
        double nrm = mean[o];
        if (recompute) {                                      // fixer_kernel: mean over years of the group means
            const int nyr = ngroups / 12;
            double acc = gacc[o];
            for (int y = 0; y < nyr; ++y)
                if (grp_len[y * 12 + m] == 0) acc += 0.0 / (double)grp_len[y * 12 + m];   // np.mean of an empty slice
            nrm = acc / nyr;
        }
        const double vv = var[o];
        const double se = vv >= 0 ? sqrt(vv) : 0.0;           // interp_tair.py:816
        fn[v][(size_t)m * P + q] = good ? (float)nrm : TWXI_FILL_F4;
        fs[v][(size_t)m * P + q] = good ? (float)se : TWXI_FILL_F4;
    }
}

int launch_tile_end(cudaStream_t s, TileState& t, const Ctx& cmin, const ChunkOut& out) {
    const int n = t.ncell * 12;
    tile_end_kernel<<<(n + 255) / 256, 256, 0, s>>>(t.ncell, cmin.ob.ngroups, cmin.ob.grp_len, t.status, t.ninv, t.mean,
                                                    t.var, t.gacc, out.norm[0], out.norm[1], out.se[0], out.se[1],
                                                    out.ninv, out.st);
    TWXI_LAUNCH_CHECK();
    return TWXI_OK;
}

}  // namespace twxi

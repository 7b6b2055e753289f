// Internal structures shared by the stage kernels of libtwxi (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <string>
#include <vector>

#include "../../include/twxi.h"

namespace twxi {

// ---- constants of the reference arithmetic ------------------------------------------------------------
// twx/utils/util_geo.py:21-22
#define TWX_RAD 0.017453292519943295
#define TWX_EARTH_KM 6371.009

void set_error(const std::string& s);
extern thread_local long long g_launches;
bool stage_timing_on();          // twxi_set_stage_timing(1): the kriging launcher brackets its ked_kernel launches with events

#define TWXI_CUDA(expr)                                                                         \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess) {                                                                \
            twxi::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                \
            return TWXI_ERR_CUDA;                                                               \
        }                                                                                       \
    } while (0)

#define TWXI_LAUNCH_CHECK()                                                                     \
    do {                                                                                        \
        ++twxi::g_launches;                                                                     \
        cudaError_t _e = cudaGetLastError();                                                    \
        if (_e != cudaSuccess) {                                                                \
            twxi::set_error(std::string("kernel launch: ") + cudaGetErrorString(_e));           \
            return TWXI_ERR_CUDA;                                                               \
        }                                                                                       \
    } while (0)

// Device view of one variable's station table (good stations, DB order).
struct StnTable {
    int n;
    const double* lon;      // degrees
    const double* lat;
    const double* elev;
    const double* tdi;
    const double* lonrad;   // lon * TWX_RAD (one IEEE multiply, same value numpy computes)
    const double* latrad;
    const double* coslat;   // cos(latrad)
    const double* lst;      // [12][n]
    const double* norm;     // [12][n]
    const double* optim;    // [12][n]
    const double* optim_anom;
    const double* nug;
    const double* psill;
    const double* rng;
    const double* gx;       // [12][n][8] station-major predictor rows per month: (1, lon, lat, elev, tdi, lst_m, norm_m, 0):
                            //         one 64-byte run per neighbour for the GWR normal equations / hat row and for the
                            //         augmented rows of the kriging system, instead of 5-6 scattered sectors
    const double* optim2;   // [n][24] station-major copy: optim_nnghs 01-12, optim_nnghs_anom 01-12 (one 192-byte run per
                            //         station instead of 24 sectors: the smoothing of a4 reads the 100 nearest stations)
    const double* vario2;   // [n][12][3] station-major copy: (nug, psill, rng) per month
    const double* H;        // [n][n] WGS-84 great-circle distance (km) between stations, rows/columns in hpos order
    const int32_t* hpos;    // [n] row/column of a station in H (Morton order of lon/lat: a point's neighbours
                            //     share 32-byte sectors of H, so the tile gather of the kriging stage reads ~3x less from L2)
};

// Device view of the observations, month-major: position p in [moff[m], moff[m+1]) holds the days of month
// m+1 in chronological order (StationSerialDataDb.mth_idx, station_data.py:576-580); day_of_pos[p] is the
// chronological day index.  obsT is station-major [n][ndays] over positions.
struct ObsTable {
    int ndays;
    int moff[13];
    const float* obsT;
    const int* day_of_pos;
    // 1981-2010 normals metadata (interp_tair.py:466-479): chronological runs of (year, month) groups
    int ngroups;               // (#years in 1981-2010 range covered) * 12, year-major
    const int* grp_start;      // [ngroups] first chronological day of the group (days are contiguous)
    const int* grp_len;        // [ngroups] number of days (0 -> mean of empty = NaN)
};

// Query batch on the device (one variable).  q indexes points; all arrays sized for `cap` points.
struct Batch {
    int npts = 0, cap = 0, k1 = 0, k1cap = 0, n_rm = 0, rm_zero = 0, ndays_cap = 0;
    int gy = 0, gx = 0;            // > 0: the points are the cells of a gy x gx grid in row-major order (work chunk)
    double *lat = nullptr, *lon = nullptr, *elev = nullptr, *tdi = nullptr, *lst = nullptr;   // lst [cap][12]
    int32_t* rm_idx = nullptr;     // [cap][TWXI_MAX_RM]
    int32_t* idx = nullptr;        // [cap][k1]
    double* dist = nullptr;        // [cap][k1]
    double* h0 = nullptr;          // [cap][k1]  WGS-84 distance point -> candidate
    int32_t* nn = nullptr;         // [cap][24]  k_norm[12], k_anom[12]
    double* vario = nullptr;       // [cap][12][3]
    double* mean = nullptr;        // [cap][12]
    double* var = nullptr;         // [cap][12]
    int32_t* status = nullptr;     // [cap] first failure code (atomicCAS from TWXI_ST_OK)
    double* daily = nullptr;       // [cap][ndays] chronological order
};

// Grow-only device scratch buffer (results that need a type/layout conversion before leaving the library, staging).
struct Scratch {
    void* p = nullptr;
    size_t bytes = 0;
    int get(void** out, size_t need) {
        if (need > bytes) {
            if (p) cudaFree(p);
            p = nullptr; bytes = 0;
            TWXI_CUDA(cudaMalloc(&p, need));
            bytes = need;
        }
        *out = p;
        return TWXI_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
};

// State of the asynchronous work-chunk call (twxi_interp_chunk_async), owned by the tmin context of the pair: results
// leave the device on a copy stream from double-buffered staging, so that the device -> host copy of chunk t overlaps the
// kernels of chunk t+1; work chunks go host -> device on their own stream into double-buffered staging, ahead of the kernels.
struct AsyncOut {
    cudaStream_t copy = nullptr;
    cudaEvent_t done = nullptr;                   // compute stream: staging of the current call written
    cudaEvent_t copied[2] = {nullptr, nullptr};   // copy stream: staging slot drained to the caller's buffers
    bool pending[2] = {false, false};
    Scratch stage[2];
    cudaStream_t h2d = nullptr;
    cudaEvent_t loaded[2] = {nullptr, nullptr};   // h2d stream: chunk staged
    cudaEvent_t unpacked[2] = {nullptr, nullptr}; // compute stream: staged chunk consumed by unpack_chunk_kernel
    bool consumed[2] = {false, false};
    bool inflight_in[2] = {false, false};         // loaded[slot] recorded and not yet waited for on the host
    Scratch win[2];
    int slot = 0, last = -1;
    long long submitted = 0;                      // chunks submitted so far
    int init();
    void destroy();
};

struct Ctx;

// A work chunk interpolated over its record in day windows (twxi_tile_begin / _days / _end), owned by the tmin context of
// the pair.  Everything the windows need is copied here at begin, so other calls on the same contexts (which reuse Batch)
// may run between windows.  Per-variable arrays are [2][...]: tmin, then tmax.
struct TileState {
    bool open = false;
    const Ctx* cmax = nullptr;
    long long gen_min = 0, gen_max = 0;  // obs generations of the pair at begin: twxi_ctx_set_obs invalidates the tile
    int ny = 0, nx = 0, ncell = 0, kh = 0, ndays = 0, next_day = 0;
    int32_t* hk = nullptr;     // [2][ncell][12] k_anom
    int32_t* hidx = nullptr;   // [2][ncell][12][kh] neighbour station indices (distance order)
    double* hz = nullptr;      // [2][ncell][12][kh] hat row z in neighbour order
    double* hoff = nullptr;    // [2][ncell][12] pt_norm - z . norm
    double* mean = nullptr;    // [2][ncell][12] kriged normals
    double* var = nullptr;     // [2][ncell][12] kriging variances
    int32_t* status = nullptr; // [ncell] status of the pair (TWXI_ST_FIXER_EMPTY is set by the first window)
    int32_t* ninv = nullptr;   // [ncell] running count of Tmin >= Tmax days
    double* carry = nullptr;   // [2][ncell][15] the last 15 fixed dailies before the next window
    double* gpart = nullptr;   // [2][ncell][32] per-lane partial sums of the open 1981-2010 (year, month) group
    double* gacc = nullptr;    // [2][ncell][12] running sums over years of the group means
    int32_t* mcarry = nullptr; // [2][ncell] int16 counts summed so far of the month run the next window continues
    bool plain_days = false;   // a twxi_tile_days window since begin: mcarry misses its days
    Scratch fixed, win, out;   // the arrays above; window dailies [2][ncell][15 + nwin + 15]; host-bound staging
    void release() { fixed.release(); win.release(); out.release(); *this = TileState(); }
};

struct KedWork;                  // ked.cu: device scratch + launch configuration of the kriging stage
struct KnnWork;                  // knn.cu: candidate lists of the gridded search
void ked_work_free(KedWork*);
void knn_work_free(KnnWork*);
int knn_mean_candidates(Ctx& c, double* out);

struct Ctx {
    int device = 0;
    cudaStream_t stream = 0;
    int n = 0;
    std::vector<void*> owned;      // device allocations freed at destroy
    StnTable st{};
    ObsTable ob{};
    bool has_obs = false;
    long long obs_gen = 0;         // number of twxi_ctx_set_obs calls
    std::vector<void*> obs_owned;
    std::vector<int> h_day_of_pos; // host copies of ob.day_of_pos / grp_start / grp_len (window position ranges)
    std::vector<int> h_grp_start, h_grp_len;
    // month runs of the whole record (twxi_tile_days_mth): maximal runs of consecutive days with one (year, month), first
    // day (ascending) and length, on the device and the host (kept out of ObsTable, which the stage kernels take by value)
    const int* mrun_start = nullptr;
    const int* mrun_len = nullptr;
    std::vector<int> h_mrun_start, h_mrun_len;
    std::string mth_error;         // why the record has no monthly means (a (year, month) in two runs); empty: it has
    double* climdivs = nullptr;
    int n_climdivs = -1;           // -1: no check
    Batch b;
    int max_optim = 0;             // largest finite optim_nnghs / optim_nnghs_anom value
    // device workspaces: owned by the context (one device, one stream), never shared between contexts
    Scratch scratch[5];
    AsyncOut async;
    TileState tile;
    KedWork* ked = nullptr;
    KnnWork* knn = nullptr;
};

// ---- stage launchers (each enqueues on ctx.stream) ----------------------------------------------------
int launch_knn(Ctx& c, int npts, const double* lat, const double* lon, const int32_t* rm_idx, int n_rm,
               int rm_zero, int k1, int32_t* idx, double* dist, double* wgt, int32_t* status, int gy = 0, int gx = 0);
int launch_nngh_params(Ctx& c, Batch& b, const int32_t* norm_override, const int32_t* anom_override, int only_mth,
                       int need_norm, int need_anom, int need_vario);
int launch_krig(Ctx& c, Batch& b, int mth, const double* vario_override);
int launch_vario_fit(Ctx& c, Batch& b, int mth);
int launch_gwr(Ctx& c, Batch& b, int mth, const double* pt_norm_override, int write_daily,
               double* out_month, int kmax, int32_t* hat_k, int32_t* hat_idx, double* hat_z);
// hat rows of all 12 months with the arithmetic of launch_gwr: [ncell][12] k and offset, [ncell][12][kh] indices and z
int launch_gwr_hat_rows(Ctx& c, Batch& b, int kh, int32_t* hk, int32_t* hidx, double* hz, double* hoff);
int launch_gwr_xval(Ctx& c, Batch& b, const int32_t* self, const int32_t* counts_host, int ncounts, double* out);
int launch_station_points(Ctx& c, Batch& b, int npts, const int32_t* sidx);
int launch_split3(cudaStream_t s, size_t n, const double* src, const int32_t* status, int per_point, double* a, double* b,
                  double* c);
int launch_build_dist_table(cudaStream_t s, int n, const double* lon, const double* lat, double* H);
int launch_station_trig(cudaStream_t s, int n, const double* lon, const double* lat, double* lonrad,
                        double* latrad, double* coslat);
int launch_unpack_chunk(cudaStream_t s, const double* wrk, int ny, int nx, const double* cd_a, int n_a,
                        const double* cd_b, int n_b, Batch& bmin, Batch& bmax);
int launch_cells_status(cudaStream_t s, int ncell, const double* climdiv, const double* cd_a, int n_a,
                        const double* cd_b, int n_b, int32_t* sa, int32_t* sb);
// Outputs of a Tmin/Tmax pair call on the ncell cells of a chunk, [v] = tmin, tmax.  A null field is not produced.
struct ChunkOut {
    int16_t* q[2] = {nullptr, nullptr};       // [ndays][ncell] quantised dailies
    float* norm[2] = {nullptr, nullptr};      // [12][ncell] normals
    float* se[2] = {nullptr, nullptr};        // [12][ncell] standard errors of the normals
    int32_t* ninv = nullptr;                  // [ncell] Tmin >= Tmax days
    uint8_t* st = nullptr;                    // [ncell] status of the pair
    float* mth[2] = {nullptr, nullptr};       // [nmth][ncell] monthly means
    size_t ncell = 0, ndays = 0, nmth = 0;
};
// f8 (twxi_interp_cells): f64 [4][ncells][12] normals of tmin, tmax, then se of tmin, tmax; may be null.
int launch_fixer(Ctx& cmin, Ctx& cmax, int ncells, int fix_invalid, int have_daily, const ChunkOut& out,
                 double* f8 = nullptr);
int launch_finalize_points(Ctx& c, Batch& b, double* daily, double* norms, double* se, double* var_out,
                           uint8_t* status);
// record.cu: the day windows of an open tile (TileState)
struct WindowSpan {
    int w0, nwin, la;          // first day, window length, look-ahead days computed past the window (<= 15)
    int p0[2][12], cnt[2][12]; // per variable and month: month-major obs positions of days w0 .. w0+nwin+la-1
    int g0, g1;                // 1981-2010 groups overlapping the window
};
int launch_tile_init(cudaStream_t s, TileState& t, const Batch& bmin, const Batch& bmax);
// A window is the GWR apply of both variables into t.win, then the fixer / quantisation from t.win.
int launch_tile_apply(cudaStream_t s, TileState& t, const Ctx& cmin, const Ctx& cmax, const WindowSpan& w);
int launch_tile_fix(cudaStream_t s, TileState& t, const Ctx& cmin, const WindowSpan& w, int16_t* qmin, int16_t* qmax);
// Month runs of the window [w0, w1) of twxi_tile_days_mth: runs g0 .. g1-1 overlap it, the first nmth of them end in it.
struct MonthSpan {
    int g0, g1, nmth;
};
int launch_tile_month(cudaStream_t s, TileState& t, const Ctx& cmin, const WindowSpan& w, const MonthSpan& m,
                      const int16_t* qmin, const int16_t* qmax, float* fmin, float* fmax);
int launch_tile_end(cudaStream_t s, TileState& t, const Ctx& cmin, const ChunkOut& out);
int launch_status_to_u8(cudaStream_t s, int n, const int32_t* in, uint8_t* out);
int launch_gather_month(cudaStream_t s, int npts, int mth0, const int32_t* st, const double* src12, double* dst);
int launch_gather_vario(cudaStream_t s, int npts, int mth0, const int32_t* st, const int32_t* nn, const double* src,
                        double* dst);

// ---- small device helpers -----------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_max_i(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// Output quantisation of step25:163-164, np.round(x, 2) / np.float32(0.01) stored into int16 (C truncation).  The
// whole-record fixer and the day windows share it: their int16 dailies are byte-identical.
__device__ __forceinline__ int16_t quantize(double x) {
    const double r = rint(x * 100.0) / 100.0;
    const double v = r / (double)0.01f;
    return (int16_t)(int)v;
}

// Haversine "a" term with the reference's operation order and no FMA contraction
// (util_geo.py:32-36): sin(dlat/2)**2 + cos(lat1)*cos(lat2)*sin(dlon/2)**2
__device__ __forceinline__ double hav_a(double lat1rad, double lon1rad, double coslat1, double lat2rad,
                                        double lon2rad, double coslat2) {
    double dlat = __dsub_rn(lat1rad, lat2rad);
    double dlon = __dsub_rn(lon1rad, lon2rad);
    double s1 = sin(dlat / 2);
    double s2 = sin(dlon / 2);
    double t = __dmul_rn(__dmul_rn(coslat1, coslat2), __dmul_rn(s2, s2));
    return __dadd_rn(__dmul_rn(s1, s1), t);
}
// util_geo.py:36-39: 6371.009 * (2 * arcsin(sqrt(a)))
__device__ __forceinline__ double hav_km(double a) {
    return __dmul_rn(TWX_EARTH_KM, __dmul_rn(2.0, asin(sqrt(a))));
}

// WGS-84 great-circle distance (km) of sp::gcdist / gstat for long-lat data (Andoyer-Lambert form; SURVEY §8c)
__device__ __forceinline__ double gcdist_sp(double lon1, double lat1, double lon2, double lat2) {
    const double DE2RA = 3.14159265358979323846 / 180.0;
    const double a = 6378.137;
    const double f = 1.0 / 298.257223563;
    const double eps = 2.220446049250313e-16;
    if (fabs(lat1 - lat2) < eps) {
        if (fabs(lon1 - lon2) < eps) return 0.0;
        if (fabs((fabs(lon1) + fabs(lon2)) - 360.0) < eps) return 0.0;
    }
    double lat1R = lat1 * DE2RA, lat2R = lat2 * DE2RA, lon1R = lon1 * DE2RA, lon2R = lon2 * DE2RA;
    double F = (lat1R + lat2R) / 2.0;
    double G = (lat1R - lat2R) / 2.0;
    double L = (lon1R - lon2R) / 2.0;
    double sG, cG, sF, cF, sL, cL;
    sincos(G, &sG, &cG);
    sincos(F, &sF, &cF);
    sincos(L, &sL, &cL);
    double sinG2 = sG * sG, cosG2 = cG * cG, sinF2 = sF * sF, cosF2 = cF * cF, sinL2 = sL * sL, cosL2 = cL * cL;
    double S = sinG2 * cosL2 + cosF2 * sinL2;
    double C = cosG2 * cosL2 + sinF2 * sinL2;
    double w = atan(sqrt(S / C));
    double R = sqrt(S * C) / w;
    double D = 2 * w * a;
    double H1 = (3 * R - 1) / (2 * C);
    double H2 = (3 * R + 1) / (2 * S);
    return D * (1 + f * H1 * sinF2 * cosG2 - f * H2 * cosF2 * sinG2);
}

// ---- FP64 tensor-pipe helpers shared by the kriging and GWR kernels ----------------------------------------------------
// mma.sync.m8n8k4.f64 ("DMMA").  C fragment: lane = 4*row + col/2 holds two adjacent columns.
__device__ __forceinline__ void dmma(double2& c, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
        : "+d"(c.x), "+d"(c.y) : "d"(a), "d"(b));
}
// c = a * b with a zero accumulator: ptxas encodes the constant as RZ, so no register pair has to be zeroed first
__device__ __forceinline__ void dmma_z(double2& c, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%4,%5};"
        : "=d"(c.x), "=d"(c.y) : "d"(a), "d"(b), "d"(0.0), "d"(0.0));
}
// c = X * Y' (no accumulator input)
__device__ __forceinline__ void dmma2_z(double2& c, const double2& x, const double2& y) {
    dmma_z(c, x.x, y.x);
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
        : "+d"(c.x), "+d"(c.y) : "d"(x.y), "d"(y.y));
}
// c += X * Y' for two 8x8 tiles in C-fragment layout (even columns, then odd columns)
__device__ __forceinline__ void dmma2(double2& c, const double2& x, const double2& y) {
    dmma(c, x.x, y.x);
    dmma(c, x.y, y.y);
}

// 1/d for a normal positive double without the slow-path branches of the IEEE division: MUFU seed (~2^-20) and one
// third-order Newton step (error ~ e^3, below 1 ulp).  Non-positive / non-finite pivots are rejected by the caller.
__device__ __forceinline__ double fast_rcp(double d) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
    const double e = fma(-d, r, 1.0);
    const double e2 = fma(e, e, e);
    return fma(r, e2, r);
}

// 1/sqrt(d) for a normal positive double: MUFU seed and one third-order step (error ~ e^3), like fast_rcp.
__device__ __forceinline__ double fast_rsqrt(double d) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
    const double e = fma(-d * y, y, 1.0);
    const double g = fma(e, 0.375, 0.5) * e;
    return fma(y, g, y);
}

// Tensor-pipe form of the pivot-tile factorisation.  With the tile in C-fragment layout, lane (r, q = k/2) owns
// M[r][k]; feeding that column (zero in the other lanes) as BOTH operands of one DMMA adds the outer product
// M[:,k] M[:,k]' to every element at once: no column broadcasts and no predicates (finished rows and columns are exactly
// zero and stay zero).  Fraction-free (Bareiss) scaling keeps the reciprocal off the serial pivot chain:
//     M <- (d_k M - M[:,k] M[:,k]') / M(k-1)_(k-1,k-1),   d_k := M(k)_kk  (pivot of LDL' = d_k / previous d).
// The inverse is accumulated TRANSPOSED, Z = inv(L)': Z[c][r] -= Z[c][k] m_rk needs column k of Z and the multipliers
// m_rk = M[r][k] / d_k, both already sitting in the lanes (r, q = k/2) that feed the DMMA — no shuffles either.
// Per pivot: one shuffle (d_k), two DMMAs, ~8 scalar FP64 ops; chain = shuffle + DMUL + DMMA.  The update of Z for
// pivot k-1 is issued after the shuffle of pivot k so that it runs in the shuffle's shadow (in-order issue).
// Returns Z scaled by the inverse square roots of the pivots (columns), i.e. the transpose of inv(chol(A)).
template <int NPIV>
__device__ __forceinline__ bool elim8_mma(double2& a, int lane) {
    const int q = lane & 3;
    bool ok = true;
    double rprev = 1.0;                                       // 1 / d_(k-1)
#pragma unroll
    for (int k = 0; k < NPIV; ++k) {
        const int kq = k >> 1;
        const double mine = (k & 1) ? a.y : a.x;
        const double e = (q == kq) ? mine : 0.0;              // M[r][k] in the lanes that own column k
        const double dk = __shfl_sync(0xffffffffu, mine, 4 * k + kq);
        ok = ok && (dk > 0.0);
        const double es = -e * rprev;
        const double piv = dk * rprev;                        // (the kernels are bound by FP64-pipe work, not by this chain)
        double2 c = make_double2(piv * a.x, piv * a.y);       // M <- (d_k M - M[:,k] M[:,k]') / previous pivot
        dmma(c, es, e);
        a = c;
        rprev = fast_rcp(dk);
    }
    a.x *= rprev; a.y *= rprev;                               // Schur complement of the first NPIV pivots
    return ok;
}

// Returns Z = transpose of inv(chol(A)) in C-fragment layout (A = the SPD tile `a`).  The seven Z updates depend on
// each other only through Z, so the scheduler is free to run them behind the pivot chain.
template <bool Z_BY_FMA = true>
__device__ __forceinline__ bool chol8_inverse_t(double2 a, double2& z, int lane) {
    const int r = lane >> 2, q = lane & 3;
    z.x = (2 * q == r) ? 1.0 : 0.0;
    z.y = (2 * q + 1 == r) ? 1.0 : 0.0;
    bool ok = true;
    double dx = 1.0, dy = 1.0;                                // LDL' pivots of columns 2q, 2q+1 (scale the columns of Z)
    double rprev = 1.0;                                       // 1 / d_(k-1)
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int kq = k >> 1;
        const double mine = (k & 1) ? a.y : a.x;
        const double e = (q == kq) ? mine : 0.0;              // M[r][k] in the lanes that own column k
        const double dk = __shfl_sync(0xffffffffu, mine, 4 * k + kq);
        ok = ok && (dk > 0.0);
        const double piv = dk * rprev;
        if (kq == q) { if (k & 1) dy = piv; else dx = piv; }
        if (k < 7) {
            const double es = -e * rprev;
            double2 c = make_double2(piv * a.x, piv * a.y);   // M <- (d_k M - M[:,k] M[:,k]') / previous pivot
            dmma(c, es, e);
            a = c;
            const double p = fast_rcp(dk);
            const double mneg = (r == k) ? 0.0 : -e * p;      // Z[c][r] -= Z[c][k] m_rk
            // rank-1 update of Z with plain FMAs: three shuffles and 2 DFMAs (4 FP64-pipe cycles) instead of one DMMA
            // (16 cycles, three quarters of it multiplying zeros) - DMMA and DFMA share the pipe that bounds the kernels
            // (the GWR kernel is bound by latency and the shuffle unit instead and keeps the DMMA form)
            if (Z_BY_FMA) {
                const double zk = __shfl_sync(0xffffffffu, (k & 1) ? z.y : z.x, (lane & ~3) | kq);
                const double m0 = __shfl_sync(0xffffffffu, mneg, 8 * q + kq);
                const double m1 = __shfl_sync(0xffffffffu, mneg, 8 * q + 4 + kq);
                z.x = fma(zk, m0, z.x);
                z.y = fma(zk, m1, z.y);
            } else {
                dmma(z, (k & 1) ? z.y : z.x, mneg);
            }
            rprev = p;
        }
    }
    z.x *= fast_rsqrt(dx);
    z.y *= fast_rsqrt(dy);
    return ok;
}

// Plain LDL' form of chol8_inverse_t: M <- M - (M[:,k] / d_k) M[:,k]' on the trailing block only (finished rows and
// columns are masked out of the operands instead of being driven to zero), and the same multipliers update Z by a second
// DMMA.  The reciprocal is on the pivot chain, but a pivot costs ~13 instructions instead of ~22 (no fraction-free
// rescaling of the tile, no shuffles for Z): the kriging kernel is bound by the instructions issued next to its DMMA
// stream, not by this chain (round 2: 41.1 -> 40.2 ms; Z by DMMA alone: 40.8).
// Returns false when a pivot is not positive (or not a number).
__device__ __forceinline__ bool chol8_inverse_ldl(double2 a, double2& z, int lane) {
    const int r = lane >> 2, q = lane & 3;
    z.x = (2 * q == r) ? 1.0 : 0.0;
    z.y = (2 * q + 1 == r) ? 1.0 : 0.0;
    double dx = 1.0, dy = 1.0;                                // pivots of columns 2q, 2q+1 (scale the columns of Z)
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int kq = k >> 1;
        const double mine = (k & 1) ? a.y : a.x;
        const double dk = __shfl_sync(0xffffffffu, mine, 4 * k + kq);
        if (kq == q) { if (k & 1) dy = dk; else dx = dk; }
        if (k < 7) {
            const double e = (q == kq && r > k) ? mine : 0.0; // M[r][k], r > k, in the lanes that own column k
            const double mneg = -e * fast_rcp(dk);            // -m_rk
            dmma(a, mneg, e);                                 // trailing block: M[r][c] -= m_rk M[c][k]
            dmma(z, (k & 1) ? z.y : z.x, mneg);               // Z[c][r] -= Z[c][k] m_rk
        }
    }
    const bool ok = (dx > 0.0) && (dy > 0.0);                 // every pivot sits in the lanes q = k/2 of all rows
    z.x *= fast_rsqrt(dx);
    z.y *= fast_rsqrt(dy);
    return __all_sync(0xffffffffu, ok);
}

}  // namespace twxi

/*
 * twxi.h — C ABI of the B200-native TopoWx interpolation hot path (libtwxi.so).
 *
 * The reference (jaredwo/topowx) has no FFI layer for this path: it is pure Python (twx.interp) with one
 * in-process foreign boundary, rpy2 -> R gstat::krige (twx/interp/interp_tair.py:916).  This header is the
 * boundary a maintainer binds with ctypes to put the CUDA path behind the unchanged twx.interp API
 * (INTEGRATION.md shows the stubs).  Each entry point cites the reference interface it replaces.
 *
 * Conventions
 *  - extern "C", plain pointers and sizes only; no Python / torch types cross the ABI.
 *  - A context (twxi_ctx) belongs to ONE temperature variable (tmin or tmax) on ONE CUDA device; it owns
 *    device copies of the "good" station table (stations with isnan(bad), interp_tair.py:483-487, in DB =
 *    station-id order) and of the observations.  The caller owns every buffer it passes.
 *  - `mem` says where the caller's query / result buffers live: TWXI_MEM_HOST or TWXI_MEM_DEVICE.
 *    Context creation and twxi_ctx_set_obs always take host pointers.
 *  - Calls on one context are serialised on its stream (twxi_ctx_set_stream, default: the legacy default
 *    stream).  Every device workspace (query batch, candidate lists, kriging scratch, staging) belongs to the
 *    context, so different contexts may be driven on different streams / devices, from one host thread or several;
 *    one context must not be used from two threads at once.  With TWXI_MEM_HOST the call returns after results are in the host buffers; with
 *    TWXI_MEM_DEVICE it returns after enqueueing (results are stream-ordered).
 *  - Return value: TWXI_OK or a negative error for API misuse / CUDA failures (twxi_last_error() has text).
 *    Per-point failures never fail the call: they are reported in a per-point status byte and the point's
 *    outputs are left at fill values, mirroring the per-cell try/except of the reference drivers
 *    (scripts/step25_mpi_interp_tair.py:154-160, scripts/step24_mpi_xval_interp.py:59-65).
 *  - Months are 1..12 in arguments named `mth`; per-month arrays are indexed 0..11.
 *  - There is no CPU fallback: every entry point runs CUDA kernels or fails.
 */
#ifndef TWXI_H
#define TWXI_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TWXI_VERSION 100

#define TWXI_OK 0
#define TWXI_ERR_ARG (-1)      /* bad argument */
#define TWXI_ERR_CUDA (-2)     /* CUDA runtime error */
#define TWXI_ERR_STATE (-3)    /* call order (e.g. daily outputs requested before twxi_ctx_set_obs) */
#define TWXI_ERR_LIMIT (-4)    /* size limit of this build exceeded */

#define TWXI_MEM_HOST 0
#define TWXI_MEM_DEVICE 1

/* per-point status byte (0 = ok).  The Python layer re-raises with the reference's messages. */
#define TWXI_ST_OK 0
#define TWXI_ST_NO_NNGHS 1      /* "Cannot determine the optimal # of neighbors to use!" interp_tair.py:252,829 */
#define TWXI_ST_NO_VARIO 2      /* "Cannot determine variogram params!"                  interp_tair.py:843     */
#define TWXI_ST_TOO_FEW_STNS 3  /* IndexError: nnghs >= #candidate stations               station_select.py:164  */
#define TWXI_ST_SINGULAR 4      /* singular / non-finite kriging or GWR system (R error, FloatingPointError);   */
                                /* two co-located stations among a point's kriging neighbours are reported here, */
                                /* and so is a kriging neighbour count below 5 (intercept + four drift columns:   */
                                /* the trend matrix X'V^-1X is singular), a GWR neighbour count below 6           */
                                /* (intercept + five trend predictors)                                            */
                                /* and a variogram fit with fewer than 7 neighbours (OLS residuals of 5 trend     */
                                /* coefficients need at least 2 degrees of freedom to carry a variogram)          */
#define TWXI_ST_FIXER_EMPTY 5   /* 'No valid tmin/tmax in window'                          interp_tair.py:192     */
#define TWXI_ST_CLIMDIV 6       /* KeyError: climate division unknown to the station DB    interp_tair.py:563     */
#define TWXI_ST_KNN_TIES 7      /* more than 512 stations at a distance <= the (k+1)-th (boundary ties; twxi_knn) */
#define TWXI_ST_LIMIT 8         /* neighbour count of the point exceeds TWXI_MAX_KRIG_NNGHS (kriging kernel limit) */
#define TWXI_ST_MASKED 255      /* chunk cell with mask == 0: not a failure, nothing computed (step25:132)      */

/* fill values of the result buffers = netCDF4.default_fillvals (step25:71-88) */
#define TWXI_FILL_I2 ((int16_t)-32767)
#define TWXI_FILL_I4 ((int32_t)-2147483647)
#define TWXI_FILL_F4 9.969209968386869e+36f
#define TWXI_FILL_F8 9.969209968386869e+36

/* neighbours examined to smooth the optimal neighbour count: DFLT_INIT_NNGHS (interp_tair.py:51) */
#define TWXI_INIT_NNGHS 100
/* limits of this build */
#define TWXI_MAX_NNGHS 255      /* largest neighbour count (k+1 candidates are kept per point)  */
#define TWXI_MAX_KRIG_NNGHS 168 /* largest kriging neighbour count (k_norm); larger -> TWXI_ST_LIMIT per point */
#define TWXI_MAX_STNS 24000     /* stations per context (kNN key table lives in shared memory)  */
#define TWXI_MAX_RM 4           /* leave-out station indices per point                          */

typedef struct twxi_ctx twxi_ctx;

/* Library version (TWXI_VERSION) and last error text of the calling thread. */
int twxi_version(void);
const char* twxi_last_error(void);

/*
 * Create the context of one variable on `device`.  Replaces what PtInterpTair.__init__ /
 * XvalTairOverall.__init__ assemble per MPI rank: StationSelect(stn_da, isnan(bad)) + KrigTair + GwrTairAnom
 * (interp_tair.py:481-505, optimize.py:566-573).  Arrays are host, float64, length n_stns (good stations
 * only, DB order); per-month tables are [12][n_stns] row-major: lstMM, normMM, optim_nnghsMM,
 * optim_nnghs_anomMM, vario_nugMM, vario_psillMM, vario_rngMM (station_data.py:104-138).  NaN = missing.
 * Also builds, on the device, the station-station WGS-84 great-circle distance table that gstat uses for
 * long/lat data (interp.R:218-221,256).
 */
int twxi_ctx_create(twxi_ctx** ctx, int device, int n_stns,
                    const double* lon, const double* lat, const double* elev, const double* tdi,
                    const double* lst, const double* norm,
                    const double* optim_nnghs, const double* optim_nnghs_anom,
                    const double* vario_nug, const double* vario_psill, const double* vario_rng);

/*
 * Attach observations: host float32 [ndays][n_stns] (DB layout "(time, station_id) f4",
 * create_db_all_stations.py:307-313; same station subset/order as the context), month[ndays] in 1..12 and
 * year[ndays] (StationSerialDataDb.days, station_data.py:571-580).  Replaces StationDataWrkChk.set_obs /
 * load_obs (interp_tair.py:1027-1097): the whole table is resident in HBM, so there is no per-chunk cache.
 * Years 1981-2010 define the normals that are recomputed after a Tmin>=Tmax fix (interp_tair.py:466-479).
 * The runs of consecutive days with one (year, month) over the whole record are the months of twxi_tile_days_mth; a
 * record in which a (year, month) falls in two runs is accepted, it only has no monthly means.
 */
int twxi_ctx_set_obs(twxi_ctx* ctx, const float* obs, int ndays, const int32_t* month, const int32_t* year);

/* Set of climate divisions known to this variable's DB (keys of _get_rgn_nnghs_dict, interp_tair.py:594-610);
 * chunk cells whose climdiv is not in the set of BOTH contexts get TWXI_ST_CLIMDIV.  Host array. */
int twxi_ctx_set_climdivs(twxi_ctx* ctx, const double* climdivs, int n);

/* CUDA stream (cudaStream_t as void*) on which this context's work is enqueued; NULL = default stream. */
int twxi_ctx_set_stream(twxi_ctx* ctx, void* cuda_stream);
int twxi_ctx_destroy(twxi_ctx* ctx);
int twxi_ctx_n_stns(const twxi_ctx* ctx);
int twxi_ctx_n_days(const twxi_ctx* ctx);

/*
 * Stage a1-a3: batched k-nearest-station search.  Replaces StationSelect.__set_pt + set_ngh_stns
 * (station_select.py:72-192) with grt_circle_dist (util_geo.py:24-40) for npts points at once.
 *   lat, lon       [npts] degrees
 *   rm_idx         [npts][n_rm] station indices to leave out (stns_rm), -1 = none; NULL if n_rm == 0
 *   rm_zero_dist   rm_zero_dist_stns flag (station_select.py:97-99)
 *   k1             candidates kept = nnghs + 1 (the (k+1)-th distance is the bandwidth, :164)
 * Outputs: the first k1 stations of the order (distance in km, station index) ascending, i.e. argsort(kind='stable') of
 * the distance vector with the distances this function returns; the caller re-sorts by station id (:179-182).  Stations
 * at one km are ordered by index even where their haversine terms differ, so the result for k1 is the first k1 entries of
 * the result for any larger k1.  TWXI_ST_KNN_TIES: more than 512 candidate stations lie at a distance <= the k1-th.
 *   out_idx  int32 [npts][k1], out_dist float64 [npts][k1] haversine km,
 *   out_wgt  float64 [npts][k1] bisquare weights (1-(d/d[k1-1])^2)^2 (:169), last entry 0; may be NULL
 *   status   uint8 [npts]
 */
int twxi_knn(twxi_ctx* ctx, int npts, const double* lat, const double* lon,
             const int32_t* rm_idx, int n_rm, int rm_zero_dist, int k1,
             int32_t* out_idx, double* out_dist, double* out_wgt, uint8_t* status, int mem);

/*
 * Point batch for the stage / fused entry points below (a "pt" of build_empty_pt(), interp_tair.py:200-213).
 * All arrays [npts] except lst [npts][12] (lstMM of THIS variable: LST night for tmin, day for tmax,
 * interp_tair.py:560-572).  rm_idx/n_rm/rm_zero_dist as in twxi_knn.
 */
typedef struct twxi_points {
    int32_t npts;
    const double* lat;
    const double* lon;
    const double* elev;
    const double* tdi;
    const double* lst;
    const int32_t* rm_idx;
    int32_t n_rm;
    int32_t rm_zero_dist;
} twxi_points;

/*
 * Stage a4-a5: smoothed neighbour counts and variogram parameters for every month.  Replaces
 * KrigTair.__get_nnghs / GwrTairAnom.__get_nnghs / KrigTair.__get_vario_params (interp_tair.py:821-851,
 * 245-259).  Outputs: nnghs_norm, nnghs_anom int32 [npts][12]; vario float64 [npts][12][3] (nug, psill, rng);
 * status uint8 [npts].
 */
int twxi_nngh_params(twxi_ctx* ctx, const twxi_points* pts, int32_t* nnghs_norm, int32_t* nnghs_anom,
                     double* vario, uint8_t* status, int mem);

/*
 * Stage a6-a7: moving-window regression kriging of the monthly normals.  Replaces KrigTair.krig
 * (interp_tair.py:853-926) and R krig_meantair -> gstat::krige (interp.R:198-270) for npts points.
 *   mth            1..12 = that month only (outputs [npts][1]); 0 = all months (outputs [npts][12])
 *   nnghs_override int32 [npts] or NULL (krig(nnghs=...)); vario_override float64 [npts][3] or NULL
 * Outputs float64: mean, var (kriging prediction variance), plus status uint8 [npts].
 * A point whose neighbour count (override or smoothed, in any requested month) is below 5 gets TWXI_ST_SINGULAR: the
 * trend has an intercept and four drift columns, so X'V^-1X is singular in exact arithmetic and there is no predictor.
 */
int twxi_krig(twxi_ctx* ctx, const twxi_points* pts, int mth,
              const int32_t* nnghs_override, const double* vario_override,
              double* mean, double* var, uint8_t* status, int mem);

/*
 * SURVEY 8f rank 3: moving-window variogram fitting.  Replaces BuildKrigParams.get_krig_params
 * (interp_tair.py:612-698) and the R function get_vario_params (interp.R:54-113: OLS residuals -> gstat sample
 * variogram in 5 km lags up to 1.4 x the neighbourhood radius -> exponential model with nugget = min(gamma) and the
 * sill fixed, range fitted with fit.method 7 weights -> GLS residuals -> second variogram and fit) for npts points.
 *   mth 1..12 = that month (vario [npts][1][3]); 0 = all months ([npts][12][3]); values (nugget, psill, range), a pure
 *   nugget is (sill, 0, 0) (interp.R:103-107); NaN for failed points.
 *   nnghs_override int32 [npts] or NULL = the smoothed optimal count (interp_tair.py:666-678)
 */
int twxi_fit_vario(twxi_ctx* ctx, const twxi_points* pts, int mth, const int32_t* nnghs_override,
                   double* vario, uint8_t* status, int mem);

/*
 * SURVEY 8f rank 2 (step 21): variogram fit + regression kriging in one step for all 12 months with a given neighbour
 * count per point.  Replaces KrigTairAll.krigall (interp_tair.py:700-768) / R krig_all (interp.R:147-159); with
 * rm_idx = the station itself and rm_zero_dist = 1 it is the body of XvalTairNorm.run_xval (optimize.py:239-266).
 * nnghs int32 [npts]; outputs float64 mean, var [npts][12], vario [npts][12][3] (may be NULL), status uint8 [npts].
 */
int twxi_krig_all(twxi_ctx* ctx, const twxi_points* pts, const int32_t* nnghs,
                  double* mean, double* var, double* vario, uint8_t* status, int mem);

/*
 * Stage a8-a9 (weights only): GWR hat rows.  For month mth (1..12) returns, per point, the neighbour count
 * k, the k neighbour indices in ascending (distance, index) order and the row z = x'(X'WX)^-1 X'W of
 * _gwr_series (interp_tair.py:1128-1140) in that same order.  idx int32 / z float64 are [npts][kmax].
 */
int twxi_gwr_hat(twxi_ctx* ctx, const twxi_points* pts, int mth, const int32_t* nnghs_override,
                 int kmax, int32_t* k, int32_t* idx, double* z, uint8_t* status, int mem);

/*
 * Stage a8-a9: GWR of the daily anomalies of month mth added to the point's normal.  Replaces
 * GwrTairAnom.gwr_mth (interp_tair.py:261-314).  pt_norm float64 [npts] is pt[normMM] (the kriged normal,
 * :433).  out float64 [npts][ndays_mth] in the order of StationSerialDataDb.mth_idx[mth].
 */
int twxi_gwr_mth(twxi_ctx* ctx, const twxi_points* pts, int mth, const int32_t* nnghs_override,
                 const double* pt_norm, double* out, uint8_t* status, int mem);

/*
 * a10 / a15: all 12 months of one variable at npts points.  Replaces InterpTair.interp
 * (interp_tair.py:396-439) and, with rm_idx = the station itself and rm_zero_dist = 1,
 * XvalTairOverall.run_interp (optimize.py:579-604).
 * Outputs: daily float64 [npts][ndays] (NULL = normals only), norms, se, var float64 [npts][12]
 * (se = sqrt(var) if var >= 0 else 0, interp_tair.py:816; var may be NULL), status uint8 [npts].
 */
int twxi_interp_points(twxi_ctx* ctx, const twxi_points* pts, double* daily, double* norms, double* se,
                       double* var, uint8_t* status, int mem);

/*
 * Cross validation of the GWR neighbour count (SURVEY 8f rank 2).  Replaces XvalTairAnom.run_xval
 * (twx/interp/optimize.py:505-545) for npts stations at once: every point IS a station of the context (stn_idx int32
 * [npts], indices into the context's table; the station record is the `pt`), it is left out of its own neighbour search
 * together with any co-located station (rm_zero_dist_stns=True, optimize.py:499), the neighbour search runs once with the
 * largest count, and for every count of nnghs (HOST array, int32 [n_counts], 6..TWXI_MAX_NNGHS) and every month the daily
 * anomalies are interpolated with GWR and compared with the station's own: bias = mean(interp - obs), mae, r2 =
 * linregress r^2.  Outputs float64 [npts][n_counts][12] (NaN for stations that fail), status uint8 [npts].
 */
int twxi_xval_anom(twxi_ctx* ctx, int npts, const int32_t* stn_idx, int n_counts, const int32_t* nnghs,
                   double* bias, double* mae, double* r2, uint8_t* status, int mem);

/*
 * a15 with its skill figures: the leave-one-out cross validation of the whole interpolation (kriged normal + GWR daily
 * anomaly) that XvalTairOverall / step 24 run (optimize.py:547-604), for npts stations at once.  Points are stations of
 * the context (stn_idx int32 [npts], context indices, as in twxi_xval_anom); each is left out of its own neighbour search
 * together with any co-located station (rm_zero_dist = 1, optimize.py:569).  Neighbour search, smoothed counts, kriging
 * and GWR run as in twxi_interp_points, so daily [npts][ndays], norms and se [npts][12] (float64) are byte-identical to
 * what twxi_interp_points returns for the same stations and leave-outs.  `daily` may be NULL: the series are then built
 * on the device, used for the statistics and never copied.
 * bias, mae, r2 float64 [npts][12] compare, over every record day of month m, x = the interpolated daily value with
 * y = the station's own observation (float32 widened to float64):
 *     bias = mean(x - y), mae = mean(|x - y|), r2 = Pearson r^2 (= scipy.stats.linregress(x, y)[2]**2),
 * the definitions of XvalTairAnom.run_xval (optimize.py:520-531) applied to the full series instead of the anomalies.
 * NaN for a station whose status is not TWXI_ST_OK, for a month without a day in the record, and in r2 when either
 * series is constant over the month (as np.corrcoef).  Failed stations keep fill values in daily / norms / se; an
 * stn_idx outside the table gives TWXI_ST_TOO_FEW_STNS for that point.  TWXI_ERR_STATE before twxi_ctx_set_obs.
 */
int twxi_xval_overall(twxi_ctx* ctx, int npts, const int32_t* stn_idx, double* daily, double* norms, double* se,
                      double* bias, double* mae, double* r2, uint8_t* status, int mem);

/*
 * a11 / a12: Tmin and Tmax at ncells points with the Tmin>=Tmax fixer.  Replaces PtInterpTair.interp_pt
 * (interp_tair.py:526-592) incl. tmin_tmax_fixer (:143-197) and the 1981-2010 normals recomputation
 * (:583-590).  lst_tmin / lst_tmax [ncells][12] are the "tminMM"/"tmaxMM" LST planes; climdiv may be NULL
 * (no check).  rm_idx_tmin / rm_idx_tmax int32 [ncells][n_rm] are the stns_rm leave-outs as indices into the
 * station table of the RESPECTIVE context (-1 = none; the two tables are different subsets of the DB, so one station
 * id maps to two different indices, interp_tair.py:565,574); both NULL when n_rm == 0.
 * Outputs float64: tmin, tmax [ncells][ndays]; norms/se [ncells][12] each; ninvalid int32; status uint8.
 */
int twxi_interp_cells(twxi_ctx* ctx_tmin, twxi_ctx* ctx_tmax, int ncells,
                      const double* lat, const double* lon, const double* elev, const double* tdi,
                      const double* climdiv, const double* lst_tmin, const double* lst_tmax,
                      const int32_t* rm_idx_tmin, const int32_t* rm_idx_tmax, int n_rm, int rm_zero_dist,
                      int fix_invalid,
                      double* tmin, double* tmax, double* tmin_norms, double* tmax_norms,
                      double* tmin_se, double* tmax_se, int32_t* ninvalid, uint8_t* status, int mem);

/*
 * a14: one work chunk, exactly the buffers of the step25 worker loop (step25:68-88,126-175).
 *   wrk_chk float64 [32][ny][nx]: planes 0 row, 1 col, 2 mask, 3 lat, 4 lon, 5 elev, 6 tdi, 7 climdiv,
 *           8-19 LST night 01-12 ("tminMM"), 20-31 LST day 01-12 ("tmaxMM") (tiling.py:205-213, step25:136-144)
 * Outputs (pre-filled by the library with the fill values, then written for every cell with mask != 0 that
 * succeeds): tmin, tmax int16 [ndays][ny][nx] = trunc(round(x,2)/float32(0.01)) (step25:163-164);
 * tmin_norm, tmax_norm, tmin_se, tmax_se float32 [12][ny][nx]; ninvalid int32 [ny][nx];
 * status uint8 [ny][nx] (TWXI_ST_MASKED where mask == 0).  tmin/tmax may both be NULL (normals only).
 */
int twxi_interp_chunk(twxi_ctx* ctx_tmin, twxi_ctx* ctx_tmax, const double* wrk_chk, int ny, int nx,
                      int16_t* tmin, int16_t* tmax, float* tmin_norm, float* tmax_norm,
                      float* tmin_se, float* tmax_se, int32_t* ninvalid, uint8_t* status, int mem);

/*
 * The same call without the final wait, for drivers that work through a list of chunks the way the step25 worker
 * loop does (results go to a writer, step25:176-196, while the next chunk is computed).  With host buffers the results
 * leave the device on a copy stream from double-buffered staging, so the device -> host copy of one chunk overlaps the
 * kernels of the next; the caller's buffers (wrk_chk included, which must be pinned for the overlap to happen) belong
 * to the library until twxi_interp_chunk_wait(ctx_tmin, 1) returns, or until TWO further chunks have been submitted on the
 * same context pair: the submission of chunk t+2 blocks the calling host thread until chunk t's work chunk has been read
 * and chunk t's results are complete in the caller's host buffers (it reuses chunk t's staging slot), so a driver may
 * cycle through three sets of pinned buffers without ever calling the wait.  Submitting chunk t+1 guarantees nothing
 * about chunk t.  twxi_interp_chunk_wait(ctx_tmin, 0) only orders ctx_tmin's stream after the last copy (for event
 * timing); with host_sync != 0 it also blocks until everything submitted so far is complete.  The staging, the copy
 * streams and the events belong to ctx_tmin; one submitting thread per context pair.  The wait also covers the
 * asynchronous tile calls (twxi_tile_begin_async and the calls after it), which share this sequence of submissions.
 */
int twxi_interp_chunk_async(twxi_ctx* ctx_tmin, twxi_ctx* ctx_tmax, const double* wrk_chk, int ny, int nx,
                            int16_t* tmin, int16_t* tmax, float* tmin_norm, float* tmax_norm,
                            float* tmin_se, float* tmax_se, int32_t* ninvalid, uint8_t* status, int mem);
int twxi_interp_chunk_wait(twxi_ctx* ctx_tmin, int host_sync);

/*
 * One work chunk over a long record in day windows (multi-decade records: twxi_interp_chunk holds the chunk's whole
 * daily record on the device, 12.4 GB per variable for a 250 x 250 tile over 1948-2015).
 *   twxi_tile_begin  everything of twxi_interp_chunk that does not depend on the day: unpack, kNN, neighbour counts,
 *                    kriging of the 12 normals and the 12 GWR hat rows of both variables.  Opens a "tile" on the pair
 *                    (state owned by ctx_tmin: 288 kh + 1 632 bytes per cell, kh = the largest neighbour count;
 *                    2.75 GB for a 250 x 250 tile at kh = 147; kept for the next tile until the context is destroyed); a new begin discards an open tile.  `mem` is the memory space of
 *                    wrk_chk.
 *   twxi_tile_days   the next `ndays` days of the record (windows are consecutive, any length >= 1, chronological):
 *                    tmin, tmax int16 [ndays][ny][nx], quantised exactly like twxi_interp_chunk.
 *   twxi_tile_end    after the last day: normals (recomputed from the fixed 1981-2010 dailies when any day was fixed),
 *                    se, ninvalid and status in the layouts of twxi_interp_chunk.  Closes the tile.
 * Concatenated in order, the windows' outputs and the end's outputs are byte-identical to twxi_interp_chunk's for every
 * partition of the record.  The tile shares no workspace with the other entry points, so other calls on the same contexts
 * may run between windows.  Errors: days / end without an open tile, end before every day was emitted, or either after
 * twxi_ctx_set_obs on one of the pair -> TWXI_ERR_STATE; more days than remain, or another ctx_tmax than at begin ->
 * TWXI_ERR_ARG.  With host buffers the call returns once the results are in them; with device buffers after enqueueing.
 * With twxi_set_stage_timing(1), twxi_get_stage_ms after twxi_tile_days holds the window's GWR apply (slot 3) and fixer /
 * quantisation (slot 4) times.
 */
int twxi_tile_begin(twxi_ctx* ctx_tmin, twxi_ctx* ctx_tmax, const double* wrk_chk, int ny, int nx, int mem);
int twxi_tile_days(twxi_ctx* ctx_tmin, twxi_ctx* ctx_tmax, int ndays, int16_t* tmin, int16_t* tmax, int mem);
int twxi_tile_end(twxi_ctx* ctx_tmin, twxi_ctx* ctx_tmax, float* tmin_norm, float* tmax_norm, float* tmin_se,
                  float* tmax_se, int32_t* ninvalid, uint8_t* status, int mem);

/*
 * Monthly means of the daily product, the third part of TopoWx next to the dailies and the normals (the reference writes
 * them in a post-processing pass over the daily tile files, write_ds_mthly / _TairAggregate, tiling.py:1080-1219).
 *   A month run is a maximal run of consecutive record days with one (year, month) as given to twxi_ctx_set_obs
 *   (ctx_tmin's record).  The monthly value of a cell, variable and run is
 *       float32( ((double)S / (double)n) * (double)0.01f )      (IEEE division and product, no contraction)
 *   with S the exact int32 sum of the run's int16 counts as twxi_tile_days emits them (after the Tmin >= Tmax fixer) and
 *   n the run's days in the record: a month the record covers in part averages the days it has.  The sum is exact, so no
 *   order and no window boundary changes it.  A cell whose status is not TWXI_ST_OK (masked, failed at begin, or failed
 *   by the fixer in the first window) gets TWXI_FILL_F4 in every month; fill counts never enter a sum.
 *   The means are of the stored int16 values, not of the f64 dailies, on purpose: the reference averages what it reads
 *   back from the daily files.  Parity with _TairAggregate is unpinned (it is not in this tree).
 * twxi_tile_days_mth = twxi_tile_days (the same daily bytes) plus the monthly means of every month run whose last day
 * falls in this window, chronological: tmin_mth, tmax_mth float32 [*nmth][ny][nx]; *nmth (host int32) = runs completed
 * (0 allowed).  A month kernel after the window's fixer adds the counts into an int32 carry [2][ny][nx] of the tile, so
 * nothing grows with the record.  Every argument is checked before any work is enqueued, and an error leaves the tile as
 * it was: the errors of twxi_tile_days; max_mth < 0, nmth NULL, month buffers NULL with max_mth > 0, more than max_mth
 * runs completed by the window, or a record in which a (year, month) falls in two runs or has more than 31 days ->
 * TWXI_ERR_ARG (twxi_ctx_set_obs and the daily calls accept such a record); a twxi_tile_days window earlier in the same
 * tile -> TWXI_ERR_STATE (the carry is valid only when every window since twxi_tile_begin went through this call).  The
 * month kernel is not a stage: stage timing reports the slots of twxi_tile_days.  Measured on a B200 at a 1 000 W power
 * limit: 0.065 ms per year window of a 250 x 250 tile, 2 % of the 1948-2015 stream (DESIGN.md section 5).
 */
int twxi_tile_days_mth(twxi_ctx* ctx_tmin, twxi_ctx* ctx_tmax, int ndays, int16_t* tmin, int16_t* tmax, int max_mth,
                       float* tmin_mth, float* tmax_mth, int32_t* nmth, int mem);

/*
 * The tile calls without the final wait, for drivers that hand each window to a writer while the next one is computed
 * (the record counterpart of twxi_interp_chunk_async).  Each takes the arguments of its synchronous twin, checks them the
 * same way before anything is enqueued, and computes the same bytes.  With host buffers:
 *   twxi_tile_begin_async     stages wrk_chk host -> device on the h2d stream of ctx_tmin, like twxi_interp_chunk_async;
 *   twxi_tile_days[_mth]_async, twxi_tile_end_async   stage their results on the device and copy them to the caller's
 *                             buffers on ctx_tmin's copy stream, so the device -> host copy of window t overlaps the
 *                             kernels of window t+1, and the copies of a tile's last windows overlap the kNN and kriging
 *                             of the next tile's begin.
 * Every successful such call takes the next slot of ctx_tmin's async sequence, which twxi_interp_chunk_async shares:
 * chunks and tile calls count as one sequence of submissions.  The caller's buffers of submission t (wrk_chk of a begin,
 * the outputs of a window or of an end) belong to the library until twxi_interp_chunk_wait(ctx_tmin, 1) returns, or until
 * TWO further submissions have been made on the same context pair: submitting t+2 blocks the calling host thread until
 * t's input has been read and t's results are complete in the caller's host buffers.  Three sets of pinned buffers
 * therefore carry an endless stream.  Submitting t+1 guarantees nothing about t.  The buffers must be pinned for the
 * overlap; pageable host buffers give the same results without it.
 * The host-side tile state advances at submission: windows may be submitted back to back, *nmth is written before
 * twxi_tile_days_mth_async returns, and twxi_tile_end_async closes the tile at once, so twxi_tile_begin_async of the next
 * tile may follow immediately.  An error returns the code and message of the synchronous twin, takes no slot and leaves
 * the tile as it was.  With device buffers (TWXI_MEM_DEVICE) the calls behave like their twins, which only enqueue, and
 * take no slot.  Stage timing reports the slots of the synchronous calls.
 */
int twxi_tile_begin_async(twxi_ctx* ctx_tmin, twxi_ctx* ctx_tmax, const double* wrk_chk, int ny, int nx, int mem);
int twxi_tile_days_async(twxi_ctx* ctx_tmin, twxi_ctx* ctx_tmax, int ndays, int16_t* tmin, int16_t* tmax, int mem);
int twxi_tile_days_mth_async(twxi_ctx* ctx_tmin, twxi_ctx* ctx_tmax, int ndays, int16_t* tmin, int16_t* tmax,
                             int max_mth, float* tmin_mth, float* tmax_mth, int32_t* nmth, int mem);
int twxi_tile_end_async(twxi_ctx* ctx_tmin, twxi_ctx* ctx_tmax, float* tmin_norm, float* tmax_norm, float* tmin_se,
                        float* tmax_se, int32_t* ninvalid, uint8_t* status, int mem);

/*
 * Instrumentation for bench.py: number of kernels this library launched on the calling thread's contexts
 * since the last reset, and per-stage device time (ms) of the most recent twxi_interp_chunk /
 * twxi_interp_cells / twxi_interp_points call when timing was enabled (stage order: knn, nngh_params, krig,
 * gwr_daily, fixer_quantise; 5 floats).  Timing adds event records only.
 */
int64_t twxi_launch_count(int reset);
int twxi_set_stage_timing(int enable);
int twxi_get_stage_ms(float* ms5);
/*
 * Device time (ms, CUDA events on the context's stream) of the ked_kernel launches alone - the kriging stage without
 * the distance-tile gather and the problem sort - summed since the last call, while stage timing is enabled.
 * bench.py divides the algorithmic FLOPs of the kriging systems by this figure for its roofline object.
 */
int twxi_get_ked_kernel_ms(float* ms);

/*
 * Instrumentation: which = 0 -> mean number of candidate stations per block of cells in the most recent gridded
 * neighbour search of this context (the N_c of SURVEY 8d's F_knn = 25 N_c; -1 when no gridded search has run).
 */
int twxi_ctx_stat(twxi_ctx* ctx, int which, double* out);

/*
 * Measured FP64 peak of `device` in TFLOP/s: tensor-core DMMA (mma.sync.m8n8k4.f64) and scalar DFMA loops.
 * bench.py uses the DMMA figure as the roofline denominator of the kriging kernel.
 */
int twxi_measure_fp64_peak(int device, double* dmma_tflops, double* dfma_tflops);

#ifdef __cplusplus
}
#endif
#endif /* TWXI_H */

// C ABI of libtwxi (include/twxi.h): context management, device workspaces and the stage pipelines.
#include <algorithm>
#include <cstring>
#include <cmath>

#include "twxi_internal.cuh"

namespace twxi {

static thread_local std::string g_error;
thread_local long long g_launches = 0;
static thread_local int g_timing = 0;
static thread_local float g_stage_ms[5] = {0, 0, 0, 0, 0};
bool stage_timing_on() { return g_timing != 0; }

void set_error(const std::string& s) { g_error = s; }

#define TWXI_ARG(cond, msg)                         \
    do {                                            \
        if (!(cond)) {                              \
            twxi::set_error(msg);                   \
            return TWXI_ERR_ARG;                    \
        }                                           \
    } while (0)
#define TWXI_TRY(expr)                              \
    do {                                            \
        int _rc = (expr);                           \
        if (_rc != TWXI_OK) return _rc;             \
    } while (0)

template <typename T>
static int dev_alloc(std::vector<void*>& owned, T** p, size_t count) {
    void* d = nullptr;
    TWXI_CUDA(cudaMalloc(&d, std::max<size_t>(count, 1) * sizeof(T)));
    owned.push_back(d);
    *p = static_cast<T*>(d);
    return TWXI_OK;
}

template <typename T>
static int dev_upload(Ctx& c, std::vector<void*>& owned, const T** p, const T* host, size_t count) {
    T* d = nullptr;
    TWXI_TRY(dev_alloc(owned, &d, count));
    TWXI_CUDA(cudaMemcpyAsync(d, host, count * sizeof(T), cudaMemcpyHostToDevice, c.stream));
    *p = d;
    return TWXI_OK;
}

template <typename T>
static int grow(T** p, size_t count) {
    if (*p) cudaFree(*p);
    *p = nullptr;
    void* d = nullptr;
    TWXI_CUDA(cudaMalloc(&d, std::max<size_t>(count, 1) * sizeof(T)));
    *p = static_cast<T*>(d);
    return TWXI_OK;
}

static void free_batch(Batch& b) {
    void* ps[] = {b.lat, b.lon, b.elev, b.tdi, b.lst, b.rm_idx, b.idx, b.dist, b.h0, b.nn, b.vario,
                  b.mean, b.var, b.status, b.daily};
    for (void* p : ps)
        if (p) cudaFree(p);
    b = Batch();
}

// Make the workspace large enough for npts points with k1 candidates (and ndays of daily output).
static int ensure_batch(Ctx& c, int npts, int k1, bool need_daily) {
    Batch& b = c.b;
    if (npts > b.cap || k1 > b.k1cap) {
        const int cap = std::max(npts, b.cap), kc = std::max(k1, b.k1cap);
        double* old_daily = b.daily;
        b.daily = nullptr;
        if (old_daily) cudaFree(old_daily);
        b.ndays_cap = 0;
        TWXI_TRY(grow(&b.lat, cap)); TWXI_TRY(grow(&b.lon, cap)); TWXI_TRY(grow(&b.elev, cap));
        TWXI_TRY(grow(&b.tdi, cap)); TWXI_TRY(grow(&b.lst, (size_t)cap * 12));
        TWXI_TRY(grow(&b.rm_idx, (size_t)cap * TWXI_MAX_RM));
        TWXI_TRY(grow(&b.idx, (size_t)cap * kc)); TWXI_TRY(grow(&b.dist, (size_t)cap * kc));
        TWXI_TRY(grow(&b.h0, (size_t)cap * kc));
        TWXI_TRY(grow(&b.nn, (size_t)cap * 24)); TWXI_TRY(grow(&b.vario, (size_t)cap * 36));
        TWXI_TRY(grow(&b.mean, (size_t)cap * 12)); TWXI_TRY(grow(&b.var, (size_t)cap * 12));
        TWXI_TRY(grow(&b.status, cap));
        b.cap = cap; b.k1cap = kc;
    }
    if (need_daily && (b.daily == nullptr || b.ndays_cap < c.ob.ndays)) {
        TWXI_TRY(grow(&b.daily, (size_t)b.cap * c.ob.ndays));
        b.ndays_cap = c.ob.ndays;
    }
    b.npts = npts; b.k1 = k1;
    return TWXI_OK;
}

static int default_k1(const Ctx& c) { return std::max(TWXI_INIT_NNGHS, c.max_optim) + 1; }

// Copy a point batch into the workspace (any memory space: UVA resolves the direction).
static int load_points(Ctx& c, const twxi_points* p, int k1, bool need_daily) {
    TWXI_ARG(p && p->npts >= 0, "bad points");
    TWXI_ARG(p->n_rm >= 0 && p->n_rm <= TWXI_MAX_RM, "n_rm out of range");
    TWXI_ARG(k1 >= 2 && k1 <= TWXI_MAX_NNGHS + 1, "neighbour count out of range");
    TWXI_TRY(ensure_batch(c, p->npts, k1, need_daily));
    Batch& b = c.b;
    const size_t n = (size_t)p->npts;
    if (n == 0) return TWXI_OK;
    TWXI_ARG(p->lat && p->lon, "lat/lon required");
    TWXI_CUDA(cudaMemcpyAsync(b.lat, p->lat, n * 8, cudaMemcpyDefault, c.stream));
    TWXI_CUDA(cudaMemcpyAsync(b.lon, p->lon, n * 8, cudaMemcpyDefault, c.stream));
    if (p->elev) TWXI_CUDA(cudaMemcpyAsync(b.elev, p->elev, n * 8, cudaMemcpyDefault, c.stream));
    if (p->tdi) TWXI_CUDA(cudaMemcpyAsync(b.tdi, p->tdi, n * 8, cudaMemcpyDefault, c.stream));
    if (p->lst) TWXI_CUDA(cudaMemcpyAsync(b.lst, p->lst, n * 96, cudaMemcpyDefault, c.stream));
    b.n_rm = p->rm_idx ? p->n_rm : 0;
    b.rm_zero = p->rm_zero_dist;
    b.gy = b.gx = 0;
    if (b.n_rm > 0)
        TWXI_CUDA(cudaMemcpyAsync(b.rm_idx, p->rm_idx, n * b.n_rm * 4, cudaMemcpyDefault, c.stream));
    TWXI_CUDA(cudaMemsetAsync(b.status, 0, n * 4, c.stream));
    return TWXI_OK;
}

static int run_knn(Ctx& c) {
    Batch& b = c.b;
    return launch_knn(c, b.npts, b.lat, b.lon, b.n_rm ? b.rm_idx : nullptr, b.n_rm, b.rm_zero, b.k1, b.idx, b.dist,
                      nullptr, b.status, b.gy, b.gx);
}

// Device time of the five stages (knn, nngh_params, krig, gwr, fixer): event i is recorded where stage i starts, event 5
// after the last.  A call whose work starts at stage `first` reports 0 for the stages before it.
struct StageTimer {
    cudaEvent_t ev[6];
    bool on = false;
    int first = 0;
    cudaStream_t s = 0;
    void begin(cudaStream_t stream, int first_stage = 0) {
        on = g_timing != 0;
        s = stream;
        first = first_stage;
        if (!on) return;
        for (int i = first; i < 6; ++i) cudaEventCreate(&ev[i]);
        cudaEventRecord(ev[first], s);
    }
    void mark(int i) { if (on) cudaEventRecord(ev[i], s); }
    void end(bool accumulate) {
        if (!on) return;
        cudaEventSynchronize(ev[5]);
        for (int i = 0; i < 5; ++i) {
            float ms = 0;
            if (i >= first) cudaEventElapsedTime(&ms, ev[i], ev[i + 1]);
            g_stage_ms[i] = accumulate ? g_stage_ms[i] + ms : ms;
        }
        for (int i = first; i < 6; ++i) cudaEventDestroy(ev[i]);
    }
};

// knn -> nngh_params -> krig -> gwr for the points already loaded in c.b.  The GWR step is the daily apply into c.b.daily
// with `daily`, none without it, or with `hat` the hat rows of variable v (0 tmin, 1 tmax) into that tile.
static int run_variable(Ctx& c, bool daily, StageTimer& t, TileState* hat = nullptr, int v = 0) {
    TWXI_TRY(run_knn(c));
    t.mark(1);
    TWXI_TRY(launch_nngh_params(c, c.b, nullptr, nullptr, 0, 1, daily ? 1 : 0, 1));
    t.mark(2);
    TWXI_TRY(launch_krig(c, c.b, 0, nullptr));
    t.mark(3);
    if (hat) {
        const size_t n12 = (size_t)v * hat->ncell * 12;
        TWXI_TRY(launch_gwr_hat_rows(c, c.b, hat->kh, hat->hk + n12, hat->hidx + n12 * hat->kh, hat->hz + n12 * hat->kh,
                                     hat->hoff + n12));
    } else if (daily) {
        TWXI_TRY(launch_gwr(c, c.b, 0, nullptr, 1, nullptr, 0, nullptr, nullptr, nullptr));
    }
    t.mark(4);
    return TWXI_OK;
}

template <typename T>
static int copy_out(cudaStream_t s, T* dst, const T* src, size_t count) {
    if (dst && count) TWXI_CUDA(cudaMemcpyAsync(dst, src, count * sizeof(T), cudaMemcpyDefault, s));
    return TWXI_OK;
}

// Calls f(field of a, the same field of b, element count) for each field of a pair's chunk outputs, in one fixed order.
template <typename A, typename B, typename F>
static int each_field(A& a, B& b, F f) {
    const size_t nc = a.ncell;
    for (int v = 0; v < 2; ++v) TWXI_TRY(f(a.q[v], b.q[v], a.ndays * nc));
    for (int v = 0; v < 2; ++v) TWXI_TRY(f(a.norm[v], b.norm[v], 12 * nc));
    for (int v = 0; v < 2; ++v) TWXI_TRY(f(a.se[v], b.se[v], 12 * nc));
    TWXI_TRY(f(a.ninv, b.ninv, nc));
    TWXI_TRY(f(a.st, b.st, nc));
    for (int v = 0; v < 2; ++v) TWXI_TRY(f(a.mth[v], b.mth[v], a.nmth * nc));
    return TWXI_OK;
}

static size_t piece_bytes(size_t bytes) { return (bytes + 255) & ~(size_t)255; }

// Device twin *d of the caller's outputs o in s: one 256-byte aligned piece for each field that o gives, null otherwise.
static int stage_out(Scratch& s, const ChunkOut& o, ChunkOut* d) {
    *d = o;
    size_t tot = 0;
    each_field(o, *d, [&](auto* src, auto*&, size_t n) {
        if (src) tot += piece_bytes(n * sizeof(*src));
        return TWXI_OK;
    });
    char* p;
    TWXI_TRY(s.get((void**)&p, tot));
    return each_field(o, *d, [&](auto* src, auto*& dst, size_t n) {
        if (src) {
            dst = reinterpret_cast<decltype(src)>(p);
            p += piece_bytes(n * sizeof(*src));
        }
        return TWXI_OK;
    });
}

// Enqueues on s the copies of the device twin d to the caller's outputs o (null and empty fields are skipped).
static int copy_out(cudaStream_t s, const ChunkOut& o, const ChunkOut& d) {
    return each_field(d, o, [&](auto* src, auto* dst, size_t n) { return copy_out(s, dst, src, n); });
}

// A pair call enqueues the work of both variables on ctx_tmin's stream: ctx_tmax's stream points there for the scope of
// the call, whichever way it returns.
struct PairStream {
    Ctx& cmax;
    cudaStream_t saved;
    PairStream(Ctx& cmin, Ctx& cmax_) : cmax(cmax_), saved(cmax_.stream) { cmax.stream = cmin.stream; }
    ~PairStream() { cmax.stream = saved; }
};

static int finish(Ctx& c, int mem) {
    if (mem == TWXI_MEM_HOST) TWXI_CUDA(cudaStreamSynchronize(c.stream));
    return TWXI_OK;
}

// End of a point entry point: the points' status converted to uint8, the outputs that `outputs` enqueues, then the status.
template <typename F>
static int status_tail(Ctx& c, int npts, uint8_t* status, int mem, F outputs) {
    uint8_t* st8;
    TWXI_TRY(c.scratch[1].get((void**)&st8, npts));
    TWXI_TRY(launch_status_to_u8(c.stream, npts, c.b.status, st8));
    TWXI_TRY(outputs());
    TWXI_TRY(copy_out(c.stream, status, st8, (size_t)npts));
    return finish(c, mem);
}

int AsyncOut::init() {
    if (copy) return TWXI_OK;
    TWXI_CUDA(cudaStreamCreateWithFlags(&copy, cudaStreamNonBlocking));
    TWXI_CUDA(cudaStreamCreateWithFlags(&h2d, cudaStreamNonBlocking));
    TWXI_CUDA(cudaEventCreateWithFlags(&done, cudaEventDisableTiming));
    for (int i = 0; i < 2; ++i) {
        TWXI_CUDA(cudaEventCreateWithFlags(&copied[i], cudaEventDisableTiming));
        TWXI_CUDA(cudaEventCreateWithFlags(&loaded[i], cudaEventDisableTiming));
        TWXI_CUDA(cudaEventCreateWithFlags(&unpacked[i], cudaEventDisableTiming));
    }
    return TWXI_OK;
}
void AsyncOut::destroy() {
    for (int i = 0; i < 2; ++i) {
        if (copied[i]) cudaEventDestroy(copied[i]);
        if (loaded[i]) cudaEventDestroy(loaded[i]);
        if (unpacked[i]) cudaEventDestroy(unpacked[i]);
        stage[i].release();
        win[i].release();
    }
    if (done) cudaEventDestroy(done);
    if (copy) cudaStreamDestroy(copy);
    if (h2d) cudaStreamDestroy(h2d);
    *this = AsyncOut();
}

// Lay out the per-tile arrays of TileState in one allocation (256-byte aligned pieces).
static int tile_alloc(TileState& t) {
    const size_t nc = (size_t)t.ncell, nh = (size_t)2 * nc * 12 * t.kh;
    const size_t sizes[] = {2 * nc * 12 * 4, nh * 4, nh * 8, 2 * nc * 12 * 8, 2 * nc * 12 * 8, 2 * nc * 12 * 8, nc * 4,
                            nc * 4, 2 * nc * 15 * 8, 2 * nc * 32 * 8, 2 * nc * 12 * 8, 2 * nc * 4};
    size_t off[12], tot = 0;
    for (int i = 0; i < 12; ++i) { off[i] = tot; tot += (sizes[i] + 255) & ~(size_t)255; }
    char* p;
    TWXI_TRY(t.fixed.get((void**)&p, tot));
    t.hk = reinterpret_cast<int32_t*>(p + off[0]); t.hidx = reinterpret_cast<int32_t*>(p + off[1]);
    t.hz = reinterpret_cast<double*>(p + off[2]); t.hoff = reinterpret_cast<double*>(p + off[3]);
    t.mean = reinterpret_cast<double*>(p + off[4]); t.var = reinterpret_cast<double*>(p + off[5]);
    t.status = reinterpret_cast<int32_t*>(p + off[6]); t.ninv = reinterpret_cast<int32_t*>(p + off[7]);
    t.carry = reinterpret_cast<double*>(p + off[8]); t.gpart = reinterpret_cast<double*>(p + off[9]);
    t.gacc = reinterpret_cast<double*>(p + off[10]); t.mcarry = reinterpret_cast<int32_t*>(p + off[11]);
    return TWXI_OK;
}

static bool is_device_ptr(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

}  // namespace twxi

using namespace twxi;

struct twxi_ctx : public twxi::Ctx {};

extern "C" {

int twxi_version(void) { return TWXI_VERSION; }
const char* twxi_last_error(void) { return g_error.c_str(); }

int64_t twxi_launch_count(int reset) {
    long long v = g_launches;
    if (reset) g_launches = 0;
    return v;
}
int twxi_set_stage_timing(int enable) { g_timing = enable; return TWXI_OK; }
int twxi_get_stage_ms(float* ms5) {
    TWXI_ARG(ms5, "null");
    std::memcpy(ms5, g_stage_ms, sizeof(g_stage_ms));
    return TWXI_OK;
}

int twxi_ctx_create(twxi_ctx** out, int device, int n, const double* lon, const double* lat, const double* elev,
                    const double* tdi, const double* lst, const double* norm, const double* optim_nnghs,
                    const double* optim_nnghs_anom, const double* vario_nug, const double* vario_psill,
                    const double* vario_rng) {
    TWXI_ARG(out, "ctx out is null");
    TWXI_ARG(n >= 1 && n <= TWXI_MAX_STNS, "n_stns out of range (1..TWXI_MAX_STNS)");
    TWXI_ARG(lon && lat && elev && tdi && lst && norm && optim_nnghs && optim_nnghs_anom && vario_nug &&
                 vario_psill && vario_rng, "null station array");
    int ndev = 0;
    TWXI_CUDA(cudaGetDeviceCount(&ndev));
    TWXI_ARG(device >= 0 && device < ndev, "no such CUDA device");
    TWXI_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    TWXI_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        set_error("libtwxi is built for sm_100a (B200) only");
        return TWXI_ERR_CUDA;
    }
    twxi_ctx* c = new twxi_ctx();
    c->device = device;
    c->n = n;
    StnTable& st = c->st;
    st.n = n;
    int rc = TWXI_OK;
    const size_t n12 = (size_t)n * 12;
    auto up = [&](const double** p, const double* h, size_t cnt) {
        if (rc == TWXI_OK) rc = dev_upload(*c, c->owned, p, h, cnt);
    };
    up(&st.lon, lon, n); up(&st.lat, lat, n); up(&st.elev, elev, n); up(&st.tdi, tdi, n);
    up(&st.lst, lst, n12); up(&st.norm, norm, n12); up(&st.optim, optim_nnghs, n12);
    up(&st.optim_anom, optim_nnghs_anom, n12); up(&st.nug, vario_nug, n12); up(&st.psill, vario_psill, n12);
    up(&st.rng, vario_rng, n12);
    {   // station-major copies for the neighbour-count / variogram smoothing (setup.cu)
        std::vector<double> o2((size_t)n * 24), v2((size_t)n * 36);
        for (int m = 0; m < 12; ++m)
            for (int i = 0; i < n; ++i) {
                o2[(size_t)i * 24 + m] = optim_nnghs[(size_t)m * n + i];
                o2[(size_t)i * 24 + 12 + m] = optim_nnghs_anom[(size_t)m * n + i];
                v2[(size_t)i * 36 + m * 3] = vario_nug[(size_t)m * n + i];
                v2[(size_t)i * 36 + m * 3 + 1] = vario_psill[(size_t)m * n + i];
                v2[(size_t)i * 36 + m * 3 + 2] = vario_rng[(size_t)m * n + i];
            }
        std::vector<double> gx((size_t)12 * n * 8);
        for (int m = 0; m < 12; ++m)
            for (int i = 0; i < n; ++i) {
                double* g = gx.data() + ((size_t)m * n + i) * 8;
                g[0] = 1.0; g[1] = lon[i]; g[2] = lat[i]; g[3] = elev[i]; g[4] = tdi[i];
                g[5] = lst[(size_t)m * n + i]; g[6] = norm[(size_t)m * n + i]; g[7] = 0.0;
            }
        up(&st.gx, gx.data(), gx.size());
        up(&st.optim2, o2.data(), o2.size());
        up(&st.vario2, v2.data(), v2.size());
        if (rc == TWXI_OK && cudaStreamSynchronize(c->stream) != cudaSuccess) { set_error("upload failed"); rc = TWXI_ERR_CUDA; }
    }
    double *lonrad = nullptr, *latrad = nullptr, *coslat = nullptr, *H = nullptr;
    if (rc == TWXI_OK) rc = dev_alloc(c->owned, &lonrad, n);
    if (rc == TWXI_OK) rc = dev_alloc(c->owned, &latrad, n);
    if (rc == TWXI_OK) rc = dev_alloc(c->owned, &coslat, n);
    if (rc == TWXI_OK) rc = dev_alloc(c->owned, &H, (size_t)n * n);
    if (rc == TWXI_OK) rc = launch_station_trig(c->stream, n, st.lon, st.lat, lonrad, latrad, coslat);
    // station-station distance table in Morton order of (lon, lat): H[hpos[a]][hpos[b]] = gcdist(a, b), same bits as the
    // DB-ordered table (each entry is computed from the same two stations in the same argument order)
    std::vector<int32_t> hpos(n), order(n);
    std::vector<double> plon(n), plat(n);
    {
        double lo0 = lon[0], lo1 = lon[0], la0 = lat[0], la1 = lat[0];
        for (int i = 1; i < n; ++i) {
            lo0 = std::min(lo0, lon[i]); lo1 = std::max(lo1, lon[i]);
            la0 = std::min(la0, lat[i]); la1 = std::max(la1, lat[i]);
        }
        const double sx = lo1 > lo0 ? 65535.0 / (lo1 - lo0) : 0.0, sy = la1 > la0 ? 65535.0 / (la1 - la0) : 0.0;
        auto spread = [](uint32_t v) {
            v &= 0xffffu;
            v = (v | (v << 8)) & 0x00ff00ffu; v = (v | (v << 4)) & 0x0f0f0f0fu;
            v = (v | (v << 2)) & 0x33333333u; v = (v | (v << 1)) & 0x55555555u;
            return v;
        };
        std::vector<uint32_t> key(n);
        for (int i = 0; i < n; ++i) {
            const double fx = (lon[i] - lo0) * sx, fy = (lat[i] - la0) * sy;
            const uint32_t ix = std::isfinite(fx) ? (uint32_t)fx : 0u, iy = std::isfinite(fy) ? (uint32_t)fy : 0u;
            key[i] = spread(ix) | (spread(iy) << 1);
            order[i] = i;
        }
        std::stable_sort(order.begin(), order.end(), [&](int32_t x, int32_t y) { return key[x] < key[y]; });
        for (int p = 0; p < n; ++p) { hpos[order[p]] = p; plon[p] = lon[order[p]]; plat[p] = lat[order[p]]; }
    }
    const double *d_plon = nullptr, *d_plat = nullptr;
    std::vector<void*> tmp;
    if (rc == TWXI_OK) rc = dev_upload(*c, tmp, &d_plon, plon.data(), (size_t)n);
    if (rc == TWXI_OK) rc = dev_upload(*c, tmp, &d_plat, plat.data(), (size_t)n);
    if (rc == TWXI_OK) rc = dev_upload(*c, c->owned, &st.hpos, hpos.data(), (size_t)n);
    if (rc == TWXI_OK) rc = launch_build_dist_table(c->stream, n, d_plon, d_plat, H);
    if (rc == TWXI_OK && cudaStreamSynchronize(c->stream) != cudaSuccess) {
        set_error("context build failed");
        rc = TWXI_ERR_CUDA;
    }
    cudaStreamSynchronize(c->stream);
    for (void* t : tmp) cudaFree(t);
    if (rc != TWXI_OK) {
        twxi_ctx_destroy(c);
        return rc;
    }
    st.lonrad = lonrad; st.latrad = latrad; st.coslat = coslat; st.H = H;
    double mx = 0;
    for (size_t i = 0; i < n12; ++i) {
        if (std::isfinite(optim_nnghs[i])) mx = std::max(mx, optim_nnghs[i]);
        if (std::isfinite(optim_nnghs_anom[i])) mx = std::max(mx, optim_nnghs_anom[i]);
    }
    c->max_optim = (int)std::min<double>(std::ceil(mx), TWXI_MAX_NNGHS);
    *out = c;
    return TWXI_OK;
}

int twxi_ctx_destroy(twxi_ctx* c) {
    if (!c) return TWXI_OK;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (void* p : c->owned) cudaFree(p);
    for (void* p : c->obs_owned) cudaFree(p);
    if (c->climdivs) cudaFree(c->climdivs);
    free_batch(c->b);
    for (auto& sc : c->scratch) sc.release();
    c->async.destroy();
    c->tile.release();
    ked_work_free(c->ked);
    knn_work_free(c->knn);
    delete c;
    return TWXI_OK;
}

int twxi_ctx_stat(twxi_ctx* c, int which, double* out) {
    TWXI_ARG(c && out, "null argument");
    TWXI_CUDA(cudaSetDevice(c->device));
    if (which == 0) return knn_mean_candidates(*c, out);
    set_error("unknown statistic");
    return TWXI_ERR_ARG;
}

int twxi_ctx_n_stns(const twxi_ctx* c) { return c ? c->n : 0; }
int twxi_ctx_n_days(const twxi_ctx* c) { return (c && c->has_obs) ? c->ob.ndays : 0; }

int twxi_ctx_set_stream(twxi_ctx* c, void* s) {
    TWXI_ARG(c, "null ctx");
    c->stream = static_cast<cudaStream_t>(s);
    return TWXI_OK;
}

int twxi_ctx_set_climdivs(twxi_ctx* c, const double* cd, int n) {
    TWXI_ARG(c && n >= 0 && (cd || n == 0), "bad climdivs");
    TWXI_CUDA(cudaSetDevice(c->device));
    if (c->climdivs) cudaFree(c->climdivs);
    c->climdivs = nullptr;
    TWXI_CUDA(cudaMalloc((void**)&c->climdivs, std::max(n, 1) * sizeof(double)));
    if (n) TWXI_CUDA(cudaMemcpy(c->climdivs, cd, n * sizeof(double), cudaMemcpyHostToDevice));
    c->n_climdivs = n;
    return TWXI_OK;
}

int twxi_ctx_set_obs(twxi_ctx* c, const float* obs, int ndays, const int32_t* month, const int32_t* year) {
    TWXI_ARG(c && obs && month && year && ndays >= 1, "bad obs arguments");
    TWXI_ARG((long long)c->n * ndays < (1LL << 31), "n_stns * ndays must stay below 2^31 (32-bit row offsets into the obs table)");
    TWXI_CUDA(cudaSetDevice(c->device));
    TWXI_CUDA(cudaStreamSynchronize(c->stream));
    for (void* p : c->obs_owned) cudaFree(p);
    c->obs_owned.clear();
    c->has_obs = false;
    ++c->obs_gen;
    const int n = c->n;
    ObsTable& ob = c->ob;
    ob.ndays = ndays;
    // month-major positions (StationSerialDataDb.mth_idx, station_data.py:576-580)
    std::vector<int> day_of_pos;
    day_of_pos.reserve(ndays);
    for (int m = 1; m <= 12; ++m) {
        ob.moff[m - 1] = (int)day_of_pos.size();
        for (int d = 0; d < ndays; ++d) {
            TWXI_ARG(month[d] >= 1 && month[d] <= 12, "month out of range");
            if (month[d] == m) day_of_pos.push_back(d);
        }
    }
    ob.moff[12] = ndays;
    // station-major transpose in month-major day order
    std::vector<float> obsT((size_t)n * ndays);
    for (int p = 0; p < ndays; ++p) {
        const float* src = obs + (size_t)day_of_pos[p] * n;
        for (int s = 0; s < n; ++s) obsT[(size_t)s * ndays + p] = src[s];
    }
    // (year, month) groups inside 1981-2010 (PtInterpTair.__init__, interp_tair.py:466-479); days of one group
    // are contiguous in a chronological daily record
    int y0 = 0, y1 = -1;
    for (int d = 0; d < ndays; ++d)
        if (year[d] >= 1981 && year[d] <= 2010) {
            if (y1 < y0) { y0 = year[d]; y1 = year[d]; }
            y0 = std::min(y0, (int)year[d]); y1 = std::max(y1, (int)year[d]);
        }
    const int nyr = y1 >= y0 ? y1 - y0 + 1 : 0;
    std::vector<int> gstart(std::max(nyr * 12, 1), 0), glen(std::max(nyr * 12, 1), 0);
    for (int d = 0; d < ndays; ++d) {
        if (year[d] < 1981 || year[d] > 2010) continue;
        const int g = (year[d] - y0) * 12 + month[d] - 1;
        if (glen[g] == 0) gstart[g] = d;
        TWXI_ARG(gstart[g] + glen[g] == d, "days of a (year, month) must be contiguous and chronological");
        glen[g]++;
    }
    ob.ngroups = nyr * 12;
    // month runs of the whole record (twxi_tile_days_mth): maximal runs of consecutive days with one (year, month); a
    // (year, month) met in two runs leaves the record without monthly means, it is not an error of the record
    std::vector<int> rstart, rlen;
    std::vector<long long> rkey;
    for (int d = 0; d < ndays; ++d) {
        const long long key = (long long)year[d] * 16 + month[d];
        if (d == 0 || key != rkey.back()) {
            rstart.push_back(d);
            rlen.push_back(0);
            rkey.push_back(key);
        }
        rlen.back()++;
    }
    std::string mth_error;
    std::sort(rkey.begin(), rkey.end());
    if (std::adjacent_find(rkey.begin(), rkey.end()) != rkey.end())
        mth_error = "the days of a (year, month) of the record are not consecutive: monthly means need a chronological record";
    else if (*std::max_element(rlen.begin(), rlen.end()) > 31)       // keeps the int32 sums of int16 counts exact
        mth_error = "a (year, month) of the record has more than 31 days";
    const float* d_obsT; const int *d_dop, *d_gs, *d_gl, *d_rs, *d_rl;
    TWXI_TRY(dev_upload(*c, c->obs_owned, &d_obsT, obsT.data(), obsT.size()));
    TWXI_TRY(dev_upload(*c, c->obs_owned, &d_dop, day_of_pos.data(), day_of_pos.size()));
    TWXI_TRY(dev_upload(*c, c->obs_owned, &d_gs, gstart.data(), gstart.size()));
    TWXI_TRY(dev_upload(*c, c->obs_owned, &d_gl, glen.data(), glen.size()));
    TWXI_TRY(dev_upload(*c, c->obs_owned, &d_rs, rstart.data(), rstart.size()));
    TWXI_TRY(dev_upload(*c, c->obs_owned, &d_rl, rlen.data(), rlen.size()));
    TWXI_CUDA(cudaStreamSynchronize(c->stream));
    ob.obsT = d_obsT; ob.day_of_pos = d_dop; ob.grp_start = d_gs; ob.grp_len = d_gl;
    c->mrun_start = d_rs; c->mrun_len = d_rl;
    c->h_day_of_pos = std::move(day_of_pos);
    c->h_grp_start = std::move(gstart);
    c->h_grp_len = std::move(glen);
    c->h_mrun_start = std::move(rstart);
    c->h_mrun_len = std::move(rlen);
    c->mth_error = std::move(mth_error);
    c->has_obs = true;
    return TWXI_OK;
}

int twxi_knn(twxi_ctx* c, int npts, const double* lat, const double* lon, const int32_t* rm_idx, int n_rm,
             int rm_zero_dist, int k1, int32_t* out_idx, double* out_dist, double* out_wgt, uint8_t* status, int mem) {
    TWXI_ARG(c && out_idx && out_dist && status, "null argument");
    TWXI_CUDA(cudaSetDevice(c->device));
    twxi_points p{npts, lat, lon, nullptr, nullptr, nullptr, rm_idx, n_rm, rm_zero_dist};
    TWXI_TRY(load_points(*c, &p, k1, false));
    if (npts == 0) return TWXI_OK;
    Batch& b = c->b;
    double* wgt = nullptr;
    if (out_wgt) TWXI_TRY(c->scratch[0].get((void**)&wgt, (size_t)npts * k1 * 8));
    TWXI_TRY(launch_knn(*c, npts, b.lat, b.lon, b.n_rm ? b.rm_idx : nullptr, b.n_rm, b.rm_zero, k1, b.idx, b.dist,
                        wgt, b.status));
    return status_tail(*c, npts, status, mem, [&] {
        TWXI_TRY(copy_out(c->stream, out_idx, b.idx, (size_t)npts * k1));
        TWXI_TRY(copy_out(c->stream, out_dist, b.dist, (size_t)npts * k1));
        return copy_out(c->stream, out_wgt, wgt, (size_t)npts * k1);
    });
}

// k1 needed when the caller overrides neighbour counts (host arrays are scanned; device arrays use the maximum)
static int k1_for_override(const Ctx& c, const int32_t* ovr, int npts, int mem, bool need_smooth) {
    int k = need_smooth ? default_k1(c) : 2;
    if (ovr) {
        if (mem == TWXI_MEM_HOST && !is_device_ptr(ovr)) {
            int mx = 1;
            for (int i = 0; i < npts; ++i) mx = std::max(mx, (int)ovr[i]);
            k = std::max(k, std::min(mx, TWXI_MAX_NNGHS) + 1);
        } else {
            k = TWXI_MAX_NNGHS + 1;
        }
    }
    return k;
}

static int upload_override(Ctx& c, const int32_t* ovr, int npts, int slot, const int32_t** dev) {
    *dev = nullptr;
    if (!ovr) return TWXI_OK;
    int32_t* d;
    TWXI_TRY(c.scratch[slot].get((void**)&d, (size_t)npts * 4));
    TWXI_CUDA(cudaMemcpyAsync(d, ovr, (size_t)npts * 4, cudaMemcpyDefault, c.stream));
    *dev = d;
    return TWXI_OK;
}

int twxi_nngh_params(twxi_ctx* c, const twxi_points* pts, int32_t* nnghs_norm, int32_t* nnghs_anom, double* vario,
                     uint8_t* status, int mem) {
    TWXI_ARG(c && pts && status, "null argument");
    TWXI_CUDA(cudaSetDevice(c->device));
    TWXI_TRY(load_points(*c, pts, default_k1(*c), false));
    const int npts = pts->npts;
    if (npts == 0) return TWXI_OK;
    Batch& b = c->b;
    TWXI_TRY(run_knn(*c));
    TWXI_TRY(launch_nngh_params(*c, b, nullptr, nullptr, 0, 1, 1, 1));
    return status_tail(*c, npts, status, mem, [&] {
        if (nnghs_norm) TWXI_CUDA(cudaMemcpy2DAsync(nnghs_norm, 48, b.nn, 96, 48, npts, cudaMemcpyDefault, c->stream));
        if (nnghs_anom) TWXI_CUDA(cudaMemcpy2DAsync(nnghs_anom, 48, b.nn + 12, 96, 48, npts, cudaMemcpyDefault, c->stream));
        return copy_out(c->stream, vario, b.vario, (size_t)npts * 36);
    });
}

int twxi_krig(twxi_ctx* c, const twxi_points* pts, int mth, const int32_t* nnghs_override,
              const double* vario_override, double* mean, double* var, uint8_t* status, int mem) {
    TWXI_ARG(c && pts && mean && var && status, "null argument");
    TWXI_ARG(mth >= 0 && mth <= 12, "mth must be 0..12");
    TWXI_ARG(pts->elev && pts->lst, "elev and lst are required for kriging");
    TWXI_CUDA(cudaSetDevice(c->device));
    const int npts = pts->npts;
    TWXI_TRY(load_points(*c, pts, k1_for_override(*c, nnghs_override, npts, mem, nnghs_override == nullptr), false));
    if (npts == 0) return TWXI_OK;
    Batch& b = c->b;
    const int32_t* d_ovr;
    TWXI_TRY(upload_override(*c, nnghs_override, npts, 2, &d_ovr));
    double* d_vo = nullptr;
    if (vario_override) {
        TWXI_TRY(c->scratch[3].get((void**)&d_vo, (size_t)npts * 24));
        TWXI_CUDA(cudaMemcpyAsync(d_vo, vario_override, (size_t)npts * 24, cudaMemcpyDefault, c->stream));
    }
    TWXI_TRY(run_knn(*c));
    TWXI_TRY(launch_nngh_params(*c, b, d_ovr, nullptr, mth, 1, 0, vario_override ? 0 : 1));
    TWXI_TRY(launch_krig(*c, b, mth, d_vo));
    return status_tail(*c, npts, status, mem, [&] {
        double* tmp;
        const size_t cnt = (size_t)npts * (mth ? 1 : 12);
        TWXI_TRY(c->scratch[0].get((void**)&tmp, cnt * 16));
        TWXI_TRY(launch_gather_month(c->stream, npts, mth - 1, b.status, b.mean, tmp));
        TWXI_TRY(launch_gather_month(c->stream, npts, mth - 1, b.status, b.var, tmp + cnt));
        TWXI_TRY(copy_out(c->stream, mean, tmp, cnt));
        return copy_out(c->stream, var, tmp + cnt, cnt);
    });
}

// vario [npts][12][3] -> caller's [npts][12|1][3] with NaN for failed points (and for months that were not requested)
static int copy_vario(Ctx& c, int npts, int mth, double* out) {
    const int nm = mth ? 1 : 12;
    double* tmp;
    TWXI_TRY(c.scratch[0].get((void**)&tmp, (size_t)npts * nm * 3 * 8));
    TWXI_TRY(launch_gather_vario(c.stream, npts, mth - 1, c.b.status, c.b.nn, c.b.vario, tmp));
    return copy_out(c.stream, out, tmp, (size_t)npts * nm * 3);
}

int twxi_fit_vario(twxi_ctx* c, const twxi_points* pts, int mth, const int32_t* nnghs_override, double* vario,
                   uint8_t* status, int mem) {
    TWXI_ARG(c && pts && vario && status, "null argument");
    TWXI_ARG(mth >= 0 && mth <= 12, "mth must be 0..12");
    TWXI_CUDA(cudaSetDevice(c->device));
    const int npts = pts->npts;
    TWXI_TRY(load_points(*c, pts, k1_for_override(*c, nnghs_override, npts, mem, nnghs_override == nullptr), false));
    if (npts == 0) return TWXI_OK;
    Batch& b = c->b;
    const int32_t* d_ovr;
    TWXI_TRY(upload_override(*c, nnghs_override, npts, 2, &d_ovr));
    TWXI_TRY(run_knn(*c));
    TWXI_TRY(launch_nngh_params(*c, b, d_ovr, nullptr, mth, 1, 0, 0));
    TWXI_TRY(launch_vario_fit(*c, b, mth));
    return status_tail(*c, npts, status, mem, [&] { return copy_vario(*c, npts, mth, vario); });
}

int twxi_krig_all(twxi_ctx* c, const twxi_points* pts, const int32_t* nnghs, double* mean, double* var, double* vario,
                  uint8_t* status, int mem) {
    TWXI_ARG(c && pts && nnghs && mean && status, "null argument");
    TWXI_ARG(pts->elev && pts->lst, "elev and lst are required for kriging");
    TWXI_CUDA(cudaSetDevice(c->device));
    const int npts = pts->npts;
    TWXI_TRY(load_points(*c, pts, k1_for_override(*c, nnghs, npts, mem, false), false));
    if (npts == 0) return TWXI_OK;
    Batch& b = c->b;
    const int32_t* d_ovr;
    TWXI_TRY(upload_override(*c, nnghs, npts, 2, &d_ovr));
    TWXI_TRY(run_knn(*c));
    TWXI_TRY(launch_nngh_params(*c, b, d_ovr, nullptr, 0, 1, 0, 0));
    TWXI_TRY(launch_vario_fit(*c, b, 0));
    TWXI_TRY(launch_krig(*c, b, 0, nullptr));
    return status_tail(*c, npts, status, mem, [&] {
        double* tmp;
        const size_t cnt = (size_t)npts * 12;
        TWXI_TRY(c->scratch[3].get((void**)&tmp, cnt * 16));
        TWXI_TRY(launch_gather_month(c->stream, npts, -1, b.status, b.mean, tmp));
        TWXI_TRY(launch_gather_month(c->stream, npts, -1, b.status, b.var, tmp + cnt));
        TWXI_TRY(copy_out(c->stream, mean, tmp, cnt));
        TWXI_TRY(copy_out(c->stream, var, tmp + cnt, cnt));
        return vario ? copy_vario(*c, npts, 0, vario) : TWXI_OK;
    });
}

int twxi_gwr_hat(twxi_ctx* c, const twxi_points* pts, int mth, const int32_t* nnghs_override, int kmax, int32_t* k,
                 int32_t* idx, double* z, uint8_t* status, int mem) {
    TWXI_ARG(c && pts && k && idx && z && status, "null argument");
    TWXI_ARG(mth >= 1 && mth <= 12, "mth must be 1..12");
    TWXI_ARG(kmax >= 1 && kmax <= TWXI_MAX_NNGHS, "kmax out of range");
    TWXI_ARG(pts->elev && pts->tdi && pts->lst, "elev, tdi and lst are required for GWR");
    TWXI_CUDA(cudaSetDevice(c->device));
    const int npts = pts->npts;
    int k1 = k1_for_override(*c, nnghs_override, npts, mem, nnghs_override == nullptr);
    TWXI_TRY(load_points(*c, pts, k1, false));
    if (npts == 0) return TWXI_OK;
    TWXI_ARG(kmax >= k1 - 1, "kmax smaller than the largest possible neighbour count");
    Batch& b = c->b;
    const int32_t* d_ovr;
    TWXI_TRY(upload_override(*c, nnghs_override, npts, 2, &d_ovr));
    TWXI_TRY(run_knn(*c));
    TWXI_TRY(launch_nngh_params(*c, b, nullptr, d_ovr, mth, 0, 1, 0));
    char* tmp;
    const size_t nz = (size_t)npts * kmax;
    TWXI_TRY(c->scratch[0].get((void**)&tmp, nz * 12 + (size_t)npts * 4));
    double* d_z = reinterpret_cast<double*>(tmp);
    int32_t* d_idx = reinterpret_cast<int32_t*>(tmp + nz * 8);
    int32_t* d_k = reinterpret_cast<int32_t*>(tmp + nz * 12);
    TWXI_CUDA(cudaMemsetAsync(tmp, 0, nz * 12 + (size_t)npts * 4, c->stream));
    TWXI_TRY(launch_gwr(*c, b, mth, nullptr, 0, nullptr, kmax, d_k, d_idx, d_z));
    return status_tail(*c, npts, status, mem, [&] {
        TWXI_TRY(copy_out(c->stream, z, d_z, nz));
        TWXI_TRY(copy_out(c->stream, idx, d_idx, nz));
        return copy_out(c->stream, k, d_k, (size_t)npts);
    });
}

int twxi_gwr_mth(twxi_ctx* c, const twxi_points* pts, int mth, const int32_t* nnghs_override, const double* pt_norm,
                 double* out, uint8_t* status, int mem) {
    TWXI_ARG(c && pts && pt_norm && out && status, "null argument");
    TWXI_ARG(mth >= 1 && mth <= 12, "mth must be 1..12");
    TWXI_ARG(pts->elev && pts->tdi && pts->lst, "elev, tdi and lst are required for GWR");
    if (!c->has_obs) { set_error("twxi_ctx_set_obs has not been called"); return TWXI_ERR_STATE; }
    TWXI_CUDA(cudaSetDevice(c->device));
    const int npts = pts->npts;
    TWXI_TRY(load_points(*c, pts, k1_for_override(*c, nnghs_override, npts, mem, nnghs_override == nullptr), false));
    if (npts == 0) return TWXI_OK;
    Batch& b = c->b;
    const int32_t* d_ovr;
    TWXI_TRY(upload_override(*c, nnghs_override, npts, 2, &d_ovr));
    const int D = c->ob.moff[mth] - c->ob.moff[mth - 1];
    char* tmp;
    TWXI_TRY(c->scratch[0].get((void**)&tmp, (size_t)npts * D * 8 + (size_t)npts * 8));
    double* d_out = reinterpret_cast<double*>(tmp);
    double* d_ptn = d_out + (size_t)npts * D;
    TWXI_CUDA(cudaMemcpyAsync(d_ptn, pt_norm, (size_t)npts * 8, cudaMemcpyDefault, c->stream));
    TWXI_CUDA(cudaMemsetAsync(d_out, 0xff, (size_t)npts * D * 8, c->stream));   // NaN for failed points
    TWXI_TRY(run_knn(*c));
    TWXI_TRY(launch_nngh_params(*c, b, nullptr, d_ovr, mth, 0, 1, 0));
    TWXI_TRY(launch_gwr(*c, b, mth, d_ptn, 0, d_out, 0, nullptr, nullptr, nullptr));
    return status_tail(*c, npts, status, mem, [&] { return copy_out(c->stream, out, d_out, (size_t)npts * D); });
}

int twxi_xval_anom(twxi_ctx* c, int npts, const int32_t* stn_idx, int n_counts, const int32_t* nnghs, double* bias,
                   double* mae, double* r2, uint8_t* status, int mem) {
    TWXI_ARG(c && stn_idx && nnghs && bias && mae && r2 && status, "null argument");
    TWXI_ARG(npts >= 0 && n_counts >= 1 && n_counts <= 64, "bad sizes");
    if (!c->has_obs) { set_error("twxi_ctx_set_obs has not been called"); return TWXI_ERR_STATE; }
    TWXI_CUDA(cudaSetDevice(c->device));
    if (npts == 0) return TWXI_OK;
    int kmax = 0;
    for (int i = 0; i < n_counts; ++i) {
        TWXI_ARG(nnghs[i] >= 6 && nnghs[i] <= TWXI_MAX_NNGHS, "neighbour count out of range (6..TWXI_MAX_NNGHS)");
        kmax = std::max(kmax, (int)nnghs[i]);
    }
    TWXI_TRY(ensure_batch(*c, npts, kmax + 1, false));
    Batch& b = c->b;
    b.n_rm = 1; b.rm_zero = 1; b.gy = b.gx = 0;                // optimize.py:499: rm_zero_dist_stns=True, stns_rm = the station
    int32_t* d_idx;
    TWXI_TRY(c->scratch[2].get((void**)&d_idx, (size_t)npts * 4));
    TWXI_CUDA(cudaMemcpyAsync(d_idx, stn_idx, (size_t)npts * 4, cudaMemcpyDefault, c->stream));
    TWXI_TRY(launch_station_points(*c, b, npts, d_idx));
    TWXI_TRY(run_knn(*c));
    const size_t cnt = (size_t)npts * n_counts * 12;
    double* d_out;
    TWXI_TRY(c->scratch[0].get((void**)&d_out, cnt * 3 * 8 + cnt * 3 * 8));
    TWXI_CUDA(cudaMemsetAsync(d_out, 0xff, cnt * 3 * 8, c->stream));       // NaN where a system is not computed
    TWXI_TRY(launch_gwr_xval(*c, b, d_idx, nnghs, n_counts, d_out));
    double* d_split = d_out + cnt * 3;
    TWXI_TRY(launch_split3(c->stream, cnt, d_out, b.status, n_counts * 12, d_split, d_split + cnt, d_split + 2 * cnt));
    return status_tail(*c, npts, status, mem, [&] {
        TWXI_TRY(copy_out(c->stream, bias, d_split, cnt));
        TWXI_TRY(copy_out(c->stream, mae, d_split + cnt, cnt));
        return copy_out(c->stream, r2, d_split + 2 * cnt, cnt);
    });
}

int twxi_interp_points(twxi_ctx* c, const twxi_points* pts, double* daily, double* norms, double* se, double* var,
                       uint8_t* status, int mem) {
    TWXI_ARG(c && pts && norms && se && status, "null argument");
    TWXI_ARG(pts->elev && pts->tdi && pts->lst, "elev, tdi and lst are required");
    if (daily && !c->has_obs) { set_error("twxi_ctx_set_obs has not been called"); return TWXI_ERR_STATE; }
    TWXI_CUDA(cudaSetDevice(c->device));
    const int npts = pts->npts;
    TWXI_TRY(load_points(*c, pts, default_k1(*c), daily != nullptr));
    if (npts == 0) return TWXI_OK;
    Batch& b = c->b;
    StageTimer t;
    t.begin(c->stream);
    TWXI_TRY(run_variable(*c, daily != nullptr, t));
    char* tmp;
    TWXI_TRY(c->scratch[0].get((void**)&tmp, (size_t)npts * (12 * 8 * 3 + 1)));
    double* d_norms = reinterpret_cast<double*>(tmp);
    double* d_se = d_norms + (size_t)npts * 12;
    double* d_var = d_se + (size_t)npts * 12;
    uint8_t* st8 = reinterpret_cast<uint8_t*>(d_var + (size_t)npts * 12);
    TWXI_TRY(launch_finalize_points(*c, b, daily ? b.daily : nullptr, d_norms, d_se, d_var, st8));
    t.mark(5);
    TWXI_TRY(copy_out(c->stream, norms, d_norms, (size_t)npts * 12));
    TWXI_TRY(copy_out(c->stream, se, d_se, (size_t)npts * 12));
    TWXI_TRY(copy_out(c->stream, var, d_var, (size_t)npts * 12));
    TWXI_TRY(copy_out(c->stream, status, st8, (size_t)npts));
    if (daily) TWXI_TRY(copy_out(c->stream, daily, b.daily, (size_t)npts * c->ob.ndays));
    t.end(false);
    return finish(*c, mem);
}

static int check_pair(twxi_ctx* a, twxi_ctx* b, bool daily) {
    TWXI_ARG(a && b, "null ctx");
    TWXI_ARG(a->device == b->device, "tmin and tmax contexts must be on the same device");
    if (daily) {
        if (!a->has_obs || !b->has_obs) { set_error("twxi_ctx_set_obs has not been called"); return TWXI_ERR_STATE; }
        TWXI_ARG(a->ob.ndays == b->ob.ndays, "tmin and tmax observation records differ in length");
    }
    return TWXI_OK;
}

// Workspaces of both variables for the ny x nx cells of a work chunk (unpack_chunk_kernel fills them).
static int chunk_batches(Ctx& cmin, Ctx& cmax, int ny, int nx, bool need_daily) {
    for (Ctx* c : {&cmin, &cmax}) {
        TWXI_TRY(ensure_batch(*c, ny * nx, default_k1(*c), need_daily));
        c->b.n_rm = 0; c->b.rm_zero = 0;
        c->b.gy = ny; c->b.gx = nx;
    }
    return TWXI_OK;
}

int twxi_interp_cells(twxi_ctx* cmin, twxi_ctx* cmax, int ncells, const double* lat, const double* lon,
                      const double* elev, const double* tdi, const double* climdiv, const double* lst_tmin,
                      const double* lst_tmax, const int32_t* rm_idx_tmin, const int32_t* rm_idx_tmax, int n_rm,
                      int rm_zero_dist, int fix_invalid,
                      double* tmin, double* tmax, double* tmin_norms, double* tmax_norms, double* tmin_se,
                      double* tmax_se, int32_t* ninvalid, uint8_t* status, int mem) {
    TWXI_ARG(tmin && tmax && tmin_norms && tmax_norms && tmin_se && tmax_se && ninvalid && status, "null output");
    TWXI_TRY(check_pair(cmin, cmax, true));
    TWXI_CUDA(cudaSetDevice(cmin->device));
    PairStream pair(*cmin, *cmax);
    // leave-out indices are context-local: the tmin and tmax station tables are different subsets of the DB
    twxi_points pa{ncells, lat, lon, elev, tdi, lst_tmin, rm_idx_tmin, n_rm, rm_zero_dist};
    twxi_points pb{ncells, lat, lon, elev, tdi, lst_tmax, rm_idx_tmax, n_rm, rm_zero_dist};
    TWXI_TRY(load_points(*cmin, &pa, default_k1(*cmin), true));
    TWXI_TRY(load_points(*cmax, &pb, default_k1(*cmax), true));
    if (ncells == 0) return TWXI_OK;
    const int nd = cmin->ob.ndays;
    if (climdiv) {
        double* d_cd;
        TWXI_TRY(cmin->scratch[2].get((void**)&d_cd, (size_t)ncells * 8));
        TWXI_CUDA(cudaMemcpyAsync(d_cd, climdiv, (size_t)ncells * 8, cudaMemcpyDefault, cmin->stream));
        TWXI_TRY(launch_cells_status(cmin->stream, ncells, d_cd, cmin->climdivs, cmin->n_climdivs, cmax->climdivs,
                                     cmax->n_climdivs, cmin->b.status, cmax->b.status));
    }
    StageTimer ta, tb;
    ta.begin(cmin->stream);
    TWXI_TRY(run_variable(*cmin, true, ta));
    ta.mark(5);
    tb.begin(cmin->stream);
    TWXI_TRY(run_variable(*cmax, true, tb));
    const size_t n12 = (size_t)ncells * 12;
    char* tmp;
    TWXI_TRY(cmin->scratch[0].get((void**)&tmp, (size_t)ncells * (12 * 8 * 4 + 4 + 1)));
    double* d_f8 = reinterpret_cast<double*>(tmp);          // normals of tmin, tmax, then se of tmin, tmax
    ChunkOut d;
    d.ninv = reinterpret_cast<int32_t*>(d_f8 + 4 * n12);
    d.st = reinterpret_cast<uint8_t*>(d.ninv + ncells);
    TWXI_TRY(launch_fixer(*cmin, *cmax, ncells, fix_invalid, 1, d, d_f8));
    tb.mark(5);
    TWXI_TRY(copy_out(cmin->stream, tmin, cmin->b.daily, (size_t)ncells * nd));
    TWXI_TRY(copy_out(cmin->stream, tmax, cmax->b.daily, (size_t)ncells * nd));
    TWXI_TRY(copy_out(cmin->stream, tmin_norms, d_f8, n12));
    TWXI_TRY(copy_out(cmin->stream, tmax_norms, d_f8 + n12, n12));
    TWXI_TRY(copy_out(cmin->stream, tmin_se, d_f8 + 2 * n12, n12));
    TWXI_TRY(copy_out(cmin->stream, tmax_se, d_f8 + 3 * n12, n12));
    TWXI_TRY(copy_out(cmin->stream, ninvalid, d.ninv, (size_t)ncells));
    TWXI_TRY(copy_out(cmin->stream, status, d.st, (size_t)ncells));
    ta.end(false);
    tb.end(true);
    return finish(*cmin, mem);
}

static int interp_chunk_impl(twxi_ctx* cmin, twxi_ctx* cmax, const double* wrk_chk, int ny, int nx, int16_t* tmin,
                             int16_t* tmax, float* tmin_norm, float* tmax_norm, float* tmin_se, float* tmax_se,
                             int32_t* ninvalid, uint8_t* status, int mem, bool async) {
    TWXI_ARG(wrk_chk && tmin_norm && tmax_norm && tmin_se && tmax_se && ninvalid && status, "null argument");
    TWXI_ARG((tmin == nullptr) == (tmax == nullptr), "tmin and tmax must both be given or both be null");
    TWXI_ARG(ny >= 1 && nx >= 1 && (long long)ny * nx <= (1 << 24), "bad chunk size");
    const bool daily = tmin != nullptr;
    TWXI_TRY(check_pair(cmin, cmax, daily));
    TWXI_CUDA(cudaSetDevice(cmin->device));
    PairStream pair(*cmin, *cmax);
    const int ncell = ny * nx;
    TWXI_TRY(chunk_batches(*cmin, *cmax, ny, nx, daily));
    const bool host = mem != TWXI_MEM_DEVICE;
    // device staging of the chunk and of the results when the caller's buffers are on the host
    const size_t wrk_bytes = (size_t)32 * ncell * 8;
    const double* d_wrk = wrk_chk;
    const bool acopy = async && host;                    // chunk and results travel on the copy streams
    AsyncOut& ao = cmin->async;
    if (acopy) {
        TWXI_TRY(ao.init());
        const int sl = ao.slot;
        // The chunk submitted two calls ago used this slot.  Block the HOST until its work chunk has been read and its
        // results are in the caller's buffers: this is what makes "valid after two further submissions" true
        // (include/twxi.h).  The device still has the previous chunk queued, so no overlap is lost.
        if (ao.inflight_in[sl]) TWXI_CUDA(cudaEventSynchronize(ao.loaded[sl]));
        ao.inflight_in[sl] = false;
        if (ao.pending[sl]) TWXI_CUDA(cudaEventSynchronize(ao.copied[sl]));
        ao.pending[sl] = false;
        double* w;
        TWXI_TRY(ao.win[sl].get((void**)&w, wrk_bytes));
        if (ao.consumed[sl]) TWXI_CUDA(cudaStreamWaitEvent(ao.h2d, ao.unpacked[sl], 0));    // slot free again
        TWXI_CUDA(cudaMemcpyAsync(w, wrk_chk, wrk_bytes, cudaMemcpyHostToDevice, ao.h2d));
        TWXI_CUDA(cudaEventRecord(ao.loaded[sl], ao.h2d));
        ao.inflight_in[sl] = true;
        TWXI_CUDA(cudaStreamWaitEvent(cmin->stream, ao.loaded[sl], 0));
        d_wrk = w;
    } else if (host) {
        double* w;
        TWXI_TRY(cmin->scratch[2].get((void**)&w, wrk_bytes));
        TWXI_CUDA(cudaMemcpyAsync(w, wrk_chk, wrk_bytes, cudaMemcpyHostToDevice, cmin->stream));
        d_wrk = w;
    }
    const ChunkOut o{{tmin, tmax}, {tmin_norm, tmax_norm}, {tmin_se, tmax_se}, ninvalid, status, {nullptr, nullptr},
                     (size_t)ncell, daily ? (size_t)cmin->ob.ndays : 0};
    ChunkOut d = o;
    if (host) TWXI_TRY(stage_out(acopy ? ao.stage[ao.slot] : cmin->scratch[0], o, &d));
    StageTimer ta, tb;
    ta.begin(cmin->stream);
    TWXI_TRY(launch_unpack_chunk(cmin->stream, d_wrk, ny, nx, cmin->climdivs, cmin->n_climdivs, cmax->climdivs,
                                 cmax->n_climdivs, cmin->b, cmax->b));
    if (acopy) {
        TWXI_CUDA(cudaEventRecord(ao.unpacked[ao.slot], cmin->stream));
        ao.consumed[ao.slot] = true;
    }
    TWXI_TRY(run_variable(*cmin, daily, ta));
    ta.mark(5);
    tb.begin(cmin->stream);
    TWXI_TRY(run_variable(*cmax, daily, tb));
    TWXI_TRY(launch_fixer(*cmin, *cmax, ncell, 1, daily ? 1 : 0, d));
    tb.mark(5);
    if (acopy) {
        TWXI_CUDA(cudaEventRecord(ao.done, cmin->stream));
        TWXI_CUDA(cudaStreamWaitEvent(ao.copy, ao.done, 0));
        TWXI_TRY(copy_out(ao.copy, o, d));
        TWXI_CUDA(cudaEventRecord(ao.copied[ao.slot], ao.copy));
        ao.pending[ao.slot] = true;
        ao.last = ao.slot;
        ao.slot ^= 1;
        ++ao.submitted;
    } else if (host) {
        TWXI_TRY(copy_out(cmin->stream, o, d));
    }
    ta.end(false);
    tb.end(true);
    return async ? TWXI_OK : finish(*cmin, mem);
}

int twxi_interp_chunk(twxi_ctx* cmin, twxi_ctx* cmax, const double* wrk_chk, int ny, int nx, int16_t* tmin,
                      int16_t* tmax, float* tmin_norm, float* tmax_norm, float* tmin_se, float* tmax_se,
                      int32_t* ninvalid, uint8_t* status, int mem) {
    return interp_chunk_impl(cmin, cmax, wrk_chk, ny, nx, tmin, tmax, tmin_norm, tmax_norm, tmin_se, tmax_se, ninvalid,
                             status, mem, false);
}

int twxi_interp_chunk_async(twxi_ctx* cmin, twxi_ctx* cmax, const double* wrk_chk, int ny, int nx, int16_t* tmin,
                            int16_t* tmax, float* tmin_norm, float* tmax_norm, float* tmin_se, float* tmax_se,
                            int32_t* ninvalid, uint8_t* status, int mem) {
    return interp_chunk_impl(cmin, cmax, wrk_chk, ny, nx, tmin, tmax, tmin_norm, tmax_norm, tmin_se, tmax_se, ninvalid,
                             status, mem, true);
}

int twxi_tile_begin(twxi_ctx* cmin, twxi_ctx* cmax, const double* wrk_chk, int ny, int nx, int mem) {
    TWXI_ARG(wrk_chk, "null argument");
    TWXI_ARG(ny >= 1 && nx >= 1 && (long long)ny * nx <= (1 << 24), "bad chunk size");
    TWXI_TRY(check_pair(cmin, cmax, true));
    TWXI_CUDA(cudaSetDevice(cmin->device));
    cmin->tile.open = false;                                  // a new begin discards an open tile
    PairStream pair(*cmin, *cmax);
    const int ncell = ny * nx;
    TWXI_TRY(chunk_batches(*cmin, *cmax, ny, nx, false));
    const double* d_wrk = wrk_chk;
    if (mem != TWXI_MEM_DEVICE) {
        double* w;
        const size_t wrk_bytes = (size_t)32 * ncell * 8;
        TWXI_TRY(cmin->scratch[2].get((void**)&w, wrk_bytes));
        TWXI_CUDA(cudaMemcpyAsync(w, wrk_chk, wrk_bytes, cudaMemcpyHostToDevice, cmin->stream));
        d_wrk = w;
    }
    TileState& t = cmin->tile;
    t.ny = ny; t.nx = nx; t.ncell = ncell;
    t.kh = std::max(cmin->b.k1, cmax->b.k1) - 1;              // k_anom < k1 of its context
    TWXI_TRY(tile_alloc(t));
    StageTimer ta, tb;
    ta.begin(cmin->stream);
    TWXI_TRY(launch_unpack_chunk(cmin->stream, d_wrk, ny, nx, cmin->climdivs, cmin->n_climdivs, cmax->climdivs,
                                 cmax->n_climdivs, cmin->b, cmax->b));
    TWXI_TRY(run_variable(*cmin, true, ta, &t, 0));
    ta.mark(5);
    tb.begin(cmin->stream);
    TWXI_TRY(run_variable(*cmax, true, tb, &t, 1));
    TWXI_TRY(launch_tile_init(cmin->stream, t, cmin->b, cmax->b));
    tb.mark(5);
    ta.end(false);
    tb.end(true);
    t.cmax = cmax;
    t.gen_min = cmin->obs_gen; t.gen_max = cmax->obs_gen;
    t.ndays = cmin->ob.ndays;
    t.next_day = 0;
    t.plain_days = false;
    TWXI_TRY(finish(*cmin, mem));
    t.open = true;
    return TWXI_OK;
}

static int tile_check(twxi_ctx* cmin, twxi_ctx* cmax) {
    TWXI_ARG(cmin && cmax, "null ctx");
    const TileState& t = cmin->tile;
    if (!t.open) { set_error("no open tile on this context pair (twxi_tile_begin)"); return TWXI_ERR_STATE; }
    TWXI_ARG(t.cmax == cmax, "ctx_tmax differs from the one the tile was begun with");
    if (!cmin->has_obs || !cmax->has_obs || cmin->obs_gen != t.gen_min || cmax->obs_gen != t.gen_max) {
        set_error("the observation record was replaced after twxi_tile_begin");
        return TWXI_ERR_STATE;
    }
    return TWXI_OK;
}

// Month-major positions of the days [d0, d1) of month m: one contiguous run, days of a month are chronological.
static void month_positions(const Ctx& c, int m, int d0, int d1, int* p0, int* cnt) {
    const int* b = c.h_day_of_pos.data() + c.ob.moff[m];
    const int* e = c.h_day_of_pos.data() + c.ob.moff[m + 1];
    const int* lo = std::lower_bound(b, e, d0);
    const int* hi = std::lower_bound(lo, e, d1);
    *p0 = (int)(lo - c.h_day_of_pos.data());
    *cnt = (int)(hi - lo);
}

// Month runs of the days [w0, w1) (ascending run starts: the runs overlapping the window are the last one that starts at
// or before w0 up to the last one that starts before w1, and all but that last one end inside the window).
static MonthSpan month_span(const Ctx& c, int w0, int w1) {
    const std::vector<int>& st = c.h_mrun_start;
    MonthSpan m;
    m.g0 = (int)(std::upper_bound(st.begin(), st.end(), w0) - st.begin()) - 1;
    m.g1 = (int)(std::lower_bound(st.begin(), st.end(), w1) - st.begin());
    m.nmth = m.g1 - m.g0 - (st[m.g1 - 1] + c.h_mrun_len[m.g1 - 1] > w1 ? 1 : 0);
    return m;
}

// One window of the open tile into o.q; with `mth`, also the monthly means of the runs that end in it into o.mth
// (twxi_tile_days_mth).
static int tile_days_impl(twxi_ctx* cmin, twxi_ctx* cmax, int ndays, ChunkOut o, int mem,
                          const MonthSpan* mth = nullptr) {
    TileState& t = cmin->tile;
    WindowSpan w;
    w.w0 = t.next_day; w.nwin = ndays;
    const int w1 = w.w0 + ndays;
    w.la = std::min(15, t.ndays - w1);
    const Ctx* cs[2] = {cmin, cmax};
    for (int v = 0; v < 2; ++v)
        for (int m = 0; m < 12; ++m) month_positions(*cs[v], m, w.w0, w1 + w.la, &w.p0[v][m], &w.cnt[v][m]);
    w.g0 = w.g1 = 0;
    for (int g = 0; g < cmin->ob.ngroups; ++g) {
        const int gs = cmin->h_grp_start[g], len = cmin->h_grp_len[g];
        if (len == 0 || gs >= w1 || gs + len <= w.w0) continue;
        if (w.g0 == w.g1) w.g0 = g;
        w.g1 = g + 1;
    }
    o.ncell = t.ncell; o.ndays = ndays; o.nmth = mth ? mth->nmth : 0;
    ChunkOut d = o;
    if (mem != TWXI_MEM_DEVICE) TWXI_TRY(stage_out(t.out, o, &d));
    StageTimer tm;
    tm.begin(cmin->stream, 3);                                // stage slots 3 (GWR daily apply) and 4 (fixer / quantise)
    TWXI_TRY(launch_tile_apply(cmin->stream, t, *cmin, *cmax, w));
    tm.mark(4);
    TWXI_TRY(launch_tile_fix(cmin->stream, t, *cmin, w, d.q[0], d.q[1]));
    tm.mark(5);
    tm.end(false);
    if (mth) TWXI_TRY(launch_tile_month(cmin->stream, t, *cmin, w, *mth, d.q[0], d.q[1], d.mth[0], d.mth[1]));
    if (mem != TWXI_MEM_DEVICE) TWXI_TRY(copy_out(cmin->stream, o, d));
    t.next_day = w1;
    return finish(*cmin, mem);
}

int twxi_tile_days(twxi_ctx* cmin, twxi_ctx* cmax, int ndays, int16_t* tmin, int16_t* tmax, int mem) {
    TWXI_TRY(tile_check(cmin, cmax));
    TWXI_ARG(tmin && tmax, "null argument");
    TWXI_ARG(ndays >= 1 && ndays <= cmin->tile.ndays - cmin->tile.next_day, "ndays must be 1 .. the days that remain");
    TWXI_CUDA(cudaSetDevice(cmin->device));
    cmin->tile.plain_days = true;
    return tile_days_impl(cmin, cmax, ndays, ChunkOut{{tmin, tmax}}, mem);
}

int twxi_tile_days_mth(twxi_ctx* cmin, twxi_ctx* cmax, int ndays, int16_t* tmin, int16_t* tmax, int max_mth,
                       float* tmin_mth, float* tmax_mth, int32_t* nmth, int mem) {
    TWXI_TRY(tile_check(cmin, cmax));
    TWXI_ARG(tmin && tmax && nmth, "null argument");
    TWXI_ARG(ndays >= 1 && ndays <= cmin->tile.ndays - cmin->tile.next_day, "ndays must be 1 .. the days that remain");
    TWXI_ARG(max_mth >= 0, "max_mth must be >= 0");
    TWXI_ARG(max_mth == 0 || (tmin_mth && tmax_mth), "null month buffer");
    TWXI_ARG(cmin->mth_error.empty(), cmin->mth_error);
    const TileState& t = cmin->tile;
    if (t.plain_days) {
        set_error("twxi_tile_days_mth after twxi_tile_days in the same tile: the month sums miss that window");
        return TWXI_ERR_STATE;
    }
    const MonthSpan m = month_span(*cmin, t.next_day, t.next_day + ndays);
    if (m.nmth > max_mth) {
        set_error("the window completes " + std::to_string(m.nmth) + " months, more than max_mth = " +
                  std::to_string(max_mth));
        return TWXI_ERR_ARG;
    }
    TWXI_CUDA(cudaSetDevice(cmin->device));
    ChunkOut o{{tmin, tmax}};
    o.mth[0] = tmin_mth; o.mth[1] = tmax_mth;
    TWXI_TRY(tile_days_impl(cmin, cmax, ndays, o, mem, &m));
    *nmth = m.nmth;
    return TWXI_OK;
}

int twxi_tile_end(twxi_ctx* cmin, twxi_ctx* cmax, float* tmin_norm, float* tmax_norm, float* tmin_se, float* tmax_se,
                  int32_t* ninvalid, uint8_t* status, int mem) {
    TWXI_TRY(tile_check(cmin, cmax));
    TWXI_ARG(tmin_norm && tmax_norm && tmin_se && tmax_se && ninvalid && status, "null argument");
    TileState& t = cmin->tile;
    if (t.next_day != t.ndays) {
        set_error("twxi_tile_end before every day of the record was emitted");
        return TWXI_ERR_STATE;
    }
    TWXI_CUDA(cudaSetDevice(cmin->device));
    const ChunkOut o{{nullptr, nullptr}, {tmin_norm, tmax_norm}, {tmin_se, tmax_se}, ninvalid, status, {nullptr, nullptr},
                     (size_t)t.ncell};
    ChunkOut d = o;
    if (mem != TWXI_MEM_DEVICE) TWXI_TRY(stage_out(t.out, o, &d));
    TWXI_TRY(launch_tile_end(cmin->stream, t, *cmin, d));
    if (mem != TWXI_MEM_DEVICE) TWXI_TRY(copy_out(cmin->stream, o, d));
    t.open = false;
    return finish(*cmin, mem);
}

int twxi_interp_chunk_wait(twxi_ctx* cmin, int host_sync) {
    TWXI_ARG(cmin != nullptr, "null context");
    TWXI_CUDA(cudaSetDevice(cmin->device));
    AsyncOut& ao = cmin->async;
    if (ao.last >= 0) TWXI_CUDA(cudaStreamWaitEvent(cmin->stream, ao.copied[ao.last], 0));    // stream order: after the last copy
    if (host_sync) {
        TWXI_CUDA(cudaStreamSynchronize(cmin->stream));
        ao.pending[0] = ao.pending[1] = false;
        ao.consumed[0] = ao.consumed[1] = false;
        ao.inflight_in[0] = ao.inflight_in[1] = false;
        ao.last = -1;
    }
    return TWXI_OK;
}

}  // extern "C"

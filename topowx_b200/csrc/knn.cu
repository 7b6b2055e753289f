// Stage a1-a3: batched k-nearest-station search (replaces twx/interp/station_select.py:72-192 +
// twx/utils/util_geo.py:24-40).
//
// One CTA per query point.  The whole station table (lat/lon in radians, cos(lat)) is streamed from L2, the
// haversine "a" term of every station is written to a shared-memory key table (8 B per station), the
// (k+1)-th smallest key is found with an 8-pass byte-wise radix select over that table, the threshold is widened
// to the last key with the same distance in km, and only the keys <= that threshold get the asin/sqrt that turns
// "a" into kilometres; they are compacted and sorted on (km, station index).
//
// Contract: the k+1 stations returned are the first k+1 of the order (km, station index) ascending, the north_star
// tie-break, i.e. numpy argsort(kind='stable') of the distance vector, with km as this kernel computes it.  Distinct
// keys often round to the same km (sqrt halves the relative spacing), so the selection boundary is decided in km, not
// in "a": knn(k) is then a prefix of knn(k+1).  TWXI_ST_KNN_TIES: more than KNN_SEL = 512 candidate stations lie at a
// distance <= the (k+1)-th distance.
//
// Bit-exactness: the "a" term uses the reference's operation order with explicit _rn intrinsics (no FMA
// contraction).  a -> km is monotone (sqrt is correctly rounded, asin monotone up to its 1-ulp error); the widening
// takes every following key whose km is <= the threshold's, and the fast path's result is re-sorted on (km, index).
#include <algorithm>
#include <cstdlib>
#include "twxi_internal.cuh"

namespace twxi {

constexpr int KNN_THREADS = 256;
constexpr int KNN_SEL = 512;   // capacity of the compacted candidate list (k+1 <= 256 plus boundary ties)

struct KnnArgs {
    int n;
    const double* latrad;
    const double* lonrad;
    const double* coslat;
    const double* qlat;
    const double* qlon;
    const int32_t* rm_idx;
    int n_rm;
    int rm_zero;
    int k1;
    int32_t* out_idx;
    double* out_dist;
    double* out_wgt;
    int32_t* status;
    // gridded queries (work chunks): per block of KNN_BLK x KNN_BLK cells a list of candidate stations that is
    // guaranteed to contain the k1 nearest stations of every cell of the block (null = scan the whole table)
    const int32_t* cand;       // [nblocks][cand_cap]
    const int32_t* cand_cnt;   // [nblocks]; < 0: no list for this block, scan the whole table
    int cand_cap, gx, nbx, gy;
    int ntab;                  // capacity of the shared-memory key table
    int mode;                  // knn_kernel: 0 = CTA per query, 1 = CTA per block of cells with an overflowed candidate list
};

constexpr int KNN_BLK = 25;    // cells per side of a candidate block (the 250 x 250 tiles divide evenly)

__device__ __forceinline__ bool pair_less(unsigned long long ka, int ia, unsigned long long kb, int ib) {
    return ka < kb || (ka == kb && ia < ib);
}

// bitonic sort of P (power of two) (key, idx) pairs in shared memory, ascending
__device__ void bitonic_sort(unsigned long long* key, int* idx, int P) {
    for (int k = 2; k <= P; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = threadIdx.x; t < P; t += KNN_THREADS) {
                int p = t ^ j;
                if (p > t) {
                    bool asc = (t & k) == 0;
                    unsigned long long ka = key[t], kb = key[p];
                    int ia = idx[t], ib = idx[p];
                    bool sw = asc ? pair_less(kb, ib, ka, ia) : pair_less(ka, ia, kb, ib);
                    if (sw) { key[t] = kb; key[p] = ka; idx[t] = ib; idx[p] = ia; }
                }
            }
            __syncthreads();
        }
    }
}

// One query point, by the whole CTA (every thread calls it with the same q).  `smem_u64`: key table of a.ntab entries, then
// the selection arrays.
__device__ void knn_query(const KnnArgs& a, const int q, unsigned long long* smem_u64) {
    unsigned long long* keys = smem_u64;                       // [ntab]
    unsigned long long* selkey = keys + a.ntab;                // [KNN_SEL]
    int* selidx = reinterpret_cast<int*>(selkey + KNN_SEL);    // [KNN_SEL]
    unsigned* hist = reinterpret_cast<unsigned*>(selidx + KNN_SEL);   // [256]
    __shared__ unsigned long long s_prefix;
    __shared__ unsigned long long s_bkm[2];                    // fast path: km bits of ranks k1 - 1 and k1
    __shared__ unsigned s_remaining, s_cnt;

    const int tid = threadIdx.x;
    const int k1 = a.k1;
    if (a.status[q] != TWXI_ST_OK) return;                     // masked cell / earlier failure
    int n = a.n;
    const int32_t* cand = nullptr;
    if (a.cand) {
        const int b = (q / a.gx / KNN_BLK) * a.nbx + (q % a.gx) / KNN_BLK;
        const int cnt = a.cand_cnt[b];
        if (cnt >= 0) { cand = a.cand + (size_t)b * a.cand_cap; n = cnt; }
    }

    if (n < k1) {                                              // fewer stations than candidates wanted: IndexError at
        if (tid == 0) a.status[q] = TWXI_ST_TOO_FEW_STNS;      // station_select.py:164 (the select below needs n >= k1)
        return;
    }

    // ---- phase 1: haversine "a" of every station (util_geo.py:27-36) -------------------------------
    const double lat1rad = __dmul_rn(a.qlat[q], TWX_RAD);
    const double lon1rad = __dmul_rn(a.qlon[q], TWX_RAD);
    const double coslat1 = cos(lat1rad);
    int rm[TWXI_MAX_RM];
#pragma unroll
    for (int i = 0; i < TWXI_MAX_RM; ++i) rm[i] = (i < a.n_rm) ? a.rm_idx[(size_t)q * a.n_rm + i] : -1;

    for (int t = tid; t < n; t += KNN_THREADS) {
        const int s = cand ? cand[t] : t;
        double av = hav_a(lat1rad, lon1rad, coslat1, a.latrad[s], a.lonrad[s], a.coslat[s]);
        unsigned long long key = (unsigned long long)__double_as_longlong(av);
        bool removed = (a.rm_zero && av == 0.0);               // station_select.py:97-99 (d == 0 <=> a == 0)
#pragma unroll
        for (int i = 0; i < TWXI_MAX_RM; ++i) removed |= (rm[i] == s);   // :101-104
        if (removed || !(av >= 0.0)) key = ~0ull;
        keys[t] = key;
    }
    if (tid == 0) { s_prefix = 0ull; s_remaining = (unsigned)k1; s_cnt = 0u; s_bkm[0] = 0ull; s_bkm[1] = ~0ull; }
    __syncthreads();

    // ---- fast path (pruned candidate lists): at most one candidate per thread.  Every key is ranked directly by counting
    // the strictly smaller keys (one 64-bit compare per pair, broadcast reads); no select passes, no compaction, two
    // barriers.  Equal keys get equal ranks: a collision among the first k1 ranks (an exact distance tie, decided by the
    // station index) sends the query to the general path below, which sorts on (km, index).  So does a best excluded key
    // (rank k1) whose km equals that of the last selected one: the station index decides that boundary, not the key.
    bool fast_done = false;
    if (n <= KNN_THREADS) {
        const unsigned long long mk = tid < n ? keys[tid] : ~0ull;
        const int valid = __syncthreads_count(mk != ~0ull);
        if (valid < k1) {                                      // IndexError at station_select.py:164
            if (tid == 0) a.status[q] = TWXI_ST_TOO_FEW_STNS;
            return;
        }
        int rank = 0;
        int j = 0;
        for (; j + 3 < n; j += 4) {
            const unsigned long long k0 = keys[j], k1v = keys[j + 1], k2 = keys[j + 2], k3 = keys[j + 3];
            rank += (k0 < mk) + (k1v < mk) + (k2 < mk) + (k3 < mk);
        }
        for (; j < n; ++j) rank += keys[j] < mk;
        const int mi = cand ? (tid < n ? cand[tid] : 0) : tid;
        const bool mine = mk != ~0ull && rank < k1;
        if (mine) { selkey[rank] = mk; selidx[rank] = mi; }
        if (mk != ~0ull && (rank == k1 - 1 || rank == k1))    // several writers only with equal keys: the same value
            s_bkm[rank - (k1 - 1)] = (unsigned long long)__double_as_longlong(hav_km(__longlong_as_double((long long)mk)));
        __syncthreads();
        const int collide = __syncthreads_or(mine && selidx[rank] != mi);
        fast_done = !collide && s_bkm[0] != s_bkm[1];
    }
    if (!fast_done) {
    // ---- phase 2: radix select of the k1-th smallest key -----------------------------------------
    for (int pass = 0; pass < 8; ++pass) {
        const int shift = 56 - 8 * pass;
        const unsigned long long mask = pass == 0 ? 0ull : (~0ull << (shift + 8));
        hist[tid] = 0u;
        __syncthreads();
        const unsigned long long prefix = s_prefix;
        for (int s = tid; s < n; s += KNN_THREADS) {
            unsigned long long k = keys[s];
            if ((k & mask) == prefix) atomicAdd(&hist[(unsigned)(k >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (tid < 32) {
            unsigned c[8], sum = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i) { c[i] = hist[tid * 8 + i]; sum += c[i]; }
            unsigned incl = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                unsigned v = __shfl_up_sync(0xffffffffu, incl, o);
                if (tid >= o) incl += v;
            }
            unsigned excl = incl - sum;
            unsigned rem = s_remaining;
            __syncwarp();                                      // every lane has read s_remaining before one lane updates it
            if (excl < rem && rem <= incl) {
                unsigned r = rem - excl;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    if (r <= c[i]) {
                        s_prefix = prefix | ((unsigned long long)(tid * 8 + i) << shift);
                        s_remaining = r;
                        break;
                    }
                    r -= c[i];
                }
            }
        }
        __syncthreads();
    }
    unsigned long long T = s_prefix;
    if (T == ~0ull) {   // fewer than k1 candidate stations: IndexError at station_select.py:164
        if (tid == 0) a.status[q] = TWXI_ST_TOO_FEW_STNS;
        return;
    }
    // keys that differ can round to the km of the k1-th smallest key: take them all, so that (km, index) decides the
    // boundary (a few nextafter steps; every thread computes the same T)
    const double Tkm = hav_km(__longlong_as_double((long long)T));
    while (hav_km(__longlong_as_double((long long)(T + 1))) <= Tkm) ++T;

    // ---- phase 3: compact keys <= T as (km, index), sort -------------------------------------------
    for (int t = tid; t < KNN_SEL; t += KNN_THREADS) { selkey[t] = ~0ull; selidx[t] = 0x7fffffff; }
    __syncthreads();
    for (int s = tid; s < n; s += KNN_THREADS) {
        unsigned long long k = keys[s];
        if (k <= T) {
            unsigned p = atomicAdd(&s_cnt, 1u);
            if (p < (unsigned)KNN_SEL) {
                selkey[p] = (unsigned long long)__double_as_longlong(hav_km(__longlong_as_double((long long)k)));
                selidx[p] = cand ? cand[s] : s;
            }
        }
    }
    __syncthreads();
    const unsigned count_le = s_cnt;
    if (count_le > (unsigned)KNN_SEL) {
        if (tid == 0) a.status[q] = TWXI_ST_KNN_TIES;
        return;
    }
    int P = 32;
    while (P < (int)count_le) P <<= 1;
    if (count_le <= (unsigned)KNN_THREADS) {
        // rank by counting: every survivor counts the survivors that precede it in (km, index) order — no barriers,
        // broadcast shared-memory reads; pairs are distinct, so the ranks are a permutation
        unsigned long long mk = 0ull;
        int mi = 0, rank = 0;
        const bool have = tid < (int)count_le;
        if (have) {
            mk = selkey[tid]; mi = selidx[tid];
            for (int j = 0; j < (int)count_le; ++j) rank += pair_less(selkey[j], selidx[j], mk, mi) ? 1 : 0;
        }
        __syncthreads();
        if (have) { selkey[rank] = mk; selidx[rank] = mi; }
        __syncthreads();
    } else {
        bitonic_sort(selkey, selidx, P);
    }
    }   // general path

    // ---- phase 4: kilometres for the fast path's k1 survivors; verify (km, index) order -------------
    int bad = 0;
    if (fast_done && tid < k1) {
        double d = hav_km(__longlong_as_double((long long)selkey[tid]));
        selkey[tid] = (unsigned long long)__double_as_longlong(d);
    }
    __syncthreads();
    if (tid + 1 < k1) bad = !pair_less(selkey[tid], selidx[tid], selkey[tid + 1], selidx[tid + 1]);
    if (__syncthreads_or(bad)) {
        int P2 = 32;
        while (P2 < k1) P2 <<= 1;
        for (int t = k1 + tid; t < P2; t += KNN_THREADS) { selkey[t] = ~0ull; selidx[t] = 0x7fffffff; }
        __syncthreads();
        bitonic_sort(selkey, selidx, P2);
    }
    const double dbw = __longlong_as_double((long long)selkey[k1 - 1]);   // station_select.py:164
    if (tid < k1) {
        double d = __longlong_as_double((long long)selkey[tid]);
        size_t o = (size_t)q * k1 + tid;
        a.out_idx[o] = selidx[tid];
        a.out_dist[o] = d;
        if (a.out_wgt) {                                       // bisquare, station_select.py:169
            double r = d / dbw;
            double u = __dsub_rn(1.0, __dmul_rn(r, r));
            a.out_wgt[o] = __dmul_rn(u, u);
        }
    }
}

// mode 0: one CTA per query point; with candidate lists the key table holds a list (a.ntab = list capacity, a few KB: six
//         CTAs per SM instead of two at 10 000 stations) and cells of blocks whose list overflowed are left to mode 1.
// mode 1: one CTA per block of cells; only blocks whose candidate list overflowed do anything: their cells are searched
//         over the whole station table (a.ntab = a.n).
__global__ void __launch_bounds__(KNN_THREADS) knn_kernel(KnnArgs a) {
    extern __shared__ unsigned long long smem_u64[];
    if (a.mode == 0) {
        const int q = blockIdx.x;
        if (a.cand) {
            const int b = (q / a.gx / KNN_BLK) * a.nbx + (q % a.gx) / KNN_BLK;
            if (a.cand_cnt[b] < 0) return;
        }
        knn_query(a, q, smem_u64);
    } else {
        const int b = blockIdx.x;
        if (a.cand_cnt[b] >= 0) return;
        const int y0 = (b / a.nbx) * KNN_BLK, x0 = (b % a.nbx) * KNN_BLK;
        const int y1 = min(y0 + KNN_BLK, a.gy), x1 = min(x0 + KNN_BLK, a.gx);
        for (int y = y0; y < y1; ++y)
            for (int x = x0; x < x1; ++x) {
                knn_query(a, y * a.gx + x, smem_u64);
                __syncthreads();                               // the next query reuses the shared tables
            }
    }
}

// Candidate stations of one block of grid cells.  With c the block's centre cell, r_c the distance of its k1-th
// nearest station and delta the largest distance from c to a cell of the block, the triangle inequality puts the
// k1 nearest stations of every cell within r_c + 2 delta of c.  The list is a superset, so the per-cell search over it
// (same arithmetic, same (distance, index) order) returns exactly what the full scan returns.
__global__ void __launch_bounds__(KNN_THREADS) knn_candidates_kernel(KnnArgs a, int gy, int32_t* cand, int32_t* cand_cnt) {
    extern __shared__ unsigned long long smem_u64[];
    unsigned long long* keys = smem_u64;                       // [n]
    unsigned* hist = reinterpret_cast<unsigned*>(keys + a.n);  // [256]
    __shared__ unsigned long long s_prefix;
    __shared__ unsigned s_remaining, s_cnt;
    __shared__ double s_delta[KNN_THREADS / 32];
    const int tid = threadIdx.x, n = a.n, k1 = a.k1, gx = a.gx;
    const int by = blockIdx.x / a.nbx, bx = blockIdx.x % a.nbx;
    const int y0 = by * KNN_BLK, x0 = bx * KNN_BLK;
    const int y1 = min(y0 + KNN_BLK, gy), x1 = min(x0 + KNN_BLK, gx);
    const int qc = ((y0 + y1 - 1) / 2) * gx + (x0 + x1 - 1) / 2;
    const double latc = __dmul_rn(a.qlat[qc], TWX_RAD), lonc = __dmul_rn(a.qlon[qc], TWX_RAD), cosc = cos(latc);
    for (int s = tid; s < n; s += KNN_THREADS) {
        const double av = hav_a(latc, lonc, cosc, a.latrad[s], a.lonrad[s], a.coslat[s]);
        keys[s] = (av >= 0.0) ? (unsigned long long)__double_as_longlong(av) : ~0ull;
    }
    // delta: farthest cell of the block from the centre cell
    double dmax = 0.0;
    const int w = x1 - x0, cells = (y1 - y0) * w;
    for (int t = tid; t < cells; t += KNN_THREADS) {
        const int q = (y0 + t / w) * gx + x0 + t % w;
        const double la = __dmul_rn(a.qlat[q], TWX_RAD), lo = __dmul_rn(a.qlon[q], TWX_RAD);
        dmax = fmax(dmax, hav_km(hav_a(latc, lonc, cosc, la, lo, cos(la))));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) dmax = fmax(dmax, __shfl_xor_sync(0xffffffffu, dmax, o));
    if ((tid & 31) == 0) s_delta[tid >> 5] = dmax;
    if (tid == 0) { s_prefix = 0ull; s_remaining = (unsigned)k1; s_cnt = 0u; }
    __syncthreads();
    for (int pass = 0; pass < 8; ++pass) {                     // k1-th smallest key of the centre cell
        const int shift = 56 - 8 * pass;
        const unsigned long long mask = pass == 0 ? 0ull : (~0ull << (shift + 8));
        hist[tid] = 0u;
        __syncthreads();
        const unsigned long long prefix = s_prefix;
        for (int s = tid; s < n; s += KNN_THREADS) {
            const unsigned long long k = keys[s];
            if ((k & mask) == prefix) atomicAdd(&hist[(unsigned)(k >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (tid == 0) {
            unsigned rem = s_remaining, acc = 0;
            for (int b = 0; b < 256; ++b) {
                if (acc + hist[b] >= rem) { s_prefix = prefix | ((unsigned long long)b << shift); s_remaining = rem - acc; break; }
                acc += hist[b];
            }
        }
        __syncthreads();
    }
    const unsigned long long T = s_prefix;
    if (T == ~0ull) {                                          // fewer than k1 stations: every cell reports it itself
        if (tid == 0) cand_cnt[blockIdx.x] = -1;
        return;
    }
    double delta = 0.0;
    for (int i = 0; i < KNN_THREADS / 32; ++i) delta = fmax(delta, s_delta[i]);
    const double rc = hav_km(__longlong_as_double((long long)T));
    const double R = (rc + 2.0 * delta) * (1.0 + 1e-9) + 1e-6;
    int32_t* out = cand + (size_t)blockIdx.x * a.cand_cap;
    for (int s = tid; s < n; s += KNN_THREADS) {
        const unsigned long long k = keys[s];
        if (k != ~0ull && hav_km(__longlong_as_double((long long)k)) <= R) {
            const unsigned p = atomicAdd(&s_cnt, 1u);
            if (p < (unsigned)a.cand_cap) out[p] = s;
        }
    }
    __syncthreads();
    if (tid == 0) cand_cnt[blockIdx.x] = s_cnt <= (unsigned)a.cand_cap ? (int)s_cnt : -1;
}

__global__ void station_trig_kernel(int n, const double* lon, const double* lat, double* lonrad, double* latrad,
                                    double* coslat) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        double lr = __dmul_rn(lat[i], TWX_RAD);
        latrad[i] = lr;
        lonrad[i] = __dmul_rn(lon[i], TWX_RAD);
        coslat[i] = cos(lr);
    }
}

__global__ void dist_table_kernel(int n, const double* lon, const double* lat, double* H) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    int i = blockIdx.y;
    if (j < n) H[(size_t)i * n + j] = (i == j) ? 0.0 : gcdist_sp(lon[i], lat[i], lon[j], lat[j]);
}

int launch_station_trig(cudaStream_t s, int n, const double* lon, const double* lat, double* lonrad,
                        double* latrad, double* coslat) {
    station_trig_kernel<<<(n + 255) / 256, 256, 0, s>>>(n, lon, lat, lonrad, latrad, coslat);
    TWXI_LAUNCH_CHECK();
    return TWXI_OK;
}

int launch_build_dist_table(cudaStream_t s, int n, const double* lon, const double* lat, double* H) {
    dim3 grid((n + 255) / 256, n);
    dist_table_kernel<<<grid, 256, 0, s>>>(n, lon, lat, H);
    TWXI_LAUNCH_CHECK();
    return TWXI_OK;
}

struct KnnWork {                 // candidate lists of the gridded search, owned by the context
    int32_t* cand = nullptr;
    int32_t* cnt = nullptr;
    size_t cand_elems = 0, cnt_elems = 0;
    int last_blocks = 0;         // blocks of the most recent gridded search (instrumentation)
};

// mean length of the candidate lists of the most recent gridded search of this context (-1: none): twxi_ctx_stat(ctx, 0)
int knn_mean_candidates(Ctx& c, double* out) {
    *out = -1.0;
    if (!c.knn || c.knn->last_blocks <= 0) return TWXI_OK;
    std::vector<int32_t> h(c.knn->last_blocks);
    TWXI_CUDA(cudaMemcpyAsync(h.data(), c.knn->cnt, h.size() * sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
    TWXI_CUDA(cudaStreamSynchronize(c.stream));
    double s = 0;
    int m = 0;
    for (int v : h) if (v >= 0) { s += v; ++m; }
    if (m) *out = s / m;
    return TWXI_OK;
}
void knn_work_free(KnnWork* w) {
    if (!w) return;
    if (w->cand) cudaFree(w->cand);
    if (w->cnt) cudaFree(w->cnt);
    delete w;
}
constexpr int KNN_CAND_CAP = 1024;

int launch_knn(Ctx& c, int npts, const double* lat, const double* lon, const int32_t* rm_idx, int n_rm,
               int rm_zero, int k1, int32_t* idx, double* dist, double* wgt, int32_t* status, int gy, int gx) {
    if (npts <= 0) return TWXI_OK;
    KnnArgs a;
    a.n = c.n; a.latrad = c.st.latrad; a.lonrad = c.st.lonrad; a.coslat = c.st.coslat;
    a.qlat = lat; a.qlon = lon; a.rm_idx = rm_idx; a.n_rm = rm_idx ? n_rm : 0; a.rm_zero = rm_zero; a.k1 = k1;
    a.out_idx = idx; a.out_dist = dist; a.out_wgt = wgt; a.status = status;
    a.cand = nullptr; a.cand_cnt = nullptr; a.cand_cap = 0; a.gx = 0; a.nbx = 0; a.gy = 0;
    a.ntab = c.n; a.mode = 0;
    int nblocks = 0;
    // gridded queries without leave-outs: prune the station table once per block of cells
    if (gy > 0 && gx > 0 && (long long)gy * gx == npts && a.n_rm == 0 && !rm_zero && c.n > 2 * k1 && !getenv("TWXI_KNN_FULL")) {
        if (!c.knn) c.knn = new KnnWork();
        KnnWork& w = *c.knn;
        const int nby = (gy + KNN_BLK - 1) / KNN_BLK, nbx = (gx + KNN_BLK - 1) / KNN_BLK;
        int cap = std::min(c.n, KNN_CAND_CAP);
        if (const char* e = getenv("TWXI_KNN_CAP")) cap = std::max(32, std::min(cap, atoi(e)));      // tests: force list overflow
        const size_t need = (size_t)nby * nbx * cap;
        if (need > w.cand_elems) {
            if (w.cand) cudaFree(w.cand);
            w.cand = nullptr; w.cand_elems = 0;
            TWXI_CUDA(cudaMalloc((void**)&w.cand, need * sizeof(int32_t)));
            w.cand_elems = need;
        }
        if ((size_t)nby * nbx > w.cnt_elems) {
            if (w.cnt) cudaFree(w.cnt);
            w.cnt = nullptr; w.cnt_elems = 0;
            TWXI_CUDA(cudaMalloc((void**)&w.cnt, (size_t)nby * nbx * sizeof(int32_t)));
            w.cnt_elems = (size_t)nby * nbx;
        }
        a.cand_cap = cap; a.gx = gx; a.nbx = nbx; a.gy = gy;
        nblocks = nby * nbx;
        const size_t smem_c = (size_t)c.n * 8 + 256 * 4;
        TWXI_CUDA(cudaFuncSetAttribute(knn_candidates_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_c));
        knn_candidates_kernel<<<nby * nbx, KNN_THREADS, smem_c, c.stream>>>(a, gy, w.cand, w.cnt);
        TWXI_LAUNCH_CHECK();
        a.cand = w.cand; a.cand_cnt = w.cnt;
        w.last_blocks = nby * nbx;
    }
    const size_t smem_full = (size_t)c.n * 8 + KNN_SEL * 12 + 256 * 4;
    TWXI_CUDA(cudaFuncSetAttribute(knn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_full));
    if (a.cand) {
        a.ntab = a.cand_cap;                                   // per-cell search over the block's list
        knn_kernel<<<npts, KNN_THREADS, (size_t)a.ntab * 8 + KNN_SEL * 12 + 256 * 4, c.stream>>>(a);
        TWXI_LAUNCH_CHECK();
        a.ntab = c.n; a.mode = 1;                              // blocks whose list overflowed: whole table (normally none)
        knn_kernel<<<nblocks, KNN_THREADS, smem_full, c.stream>>>(a);
        TWXI_LAUNCH_CHECK();
    } else {
        knn_kernel<<<npts, KNN_THREADS, smem_full, c.stream>>>(a);
        TWXI_LAUNCH_CHECK();
    }
    return TWXI_OK;
}

}  // namespace twxi

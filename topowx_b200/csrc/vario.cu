// SURVEY §8f rank 3: moving-window variogram fitting of the regression-kriging residuals, the R function get_vario_params
// (twx/interp/rpy/interp.R:54-113) that BuildKrigParams.get_krig_params (twx/interp/interp_tair.py:612-698, step 22) and
// KrigTairAll.krigall -> krig_all (interp_tair.py:700-768, interp.R:147-159, step 21) call once per (point, month):
//   1. OLS residuals of tair ~ lon + lat + elev + lst over the n neighbours; sill = var(residuals)
//   2. gstat sample variogram of the residuals: pairs with h <= 1.4 max(neighbour distance) in 5 km lags
//      (np, mean h, gamma = sum dz^2 / 2 np per non-empty lag)
//   3. exponential model, nugget fixed at min(gamma), sill fixed, RANGE fitted by weighted least squares with gstat's
//      fit.method 7 weights np / h^2 (Gauss-Newton from 0.1 max h); pure nugget where the fit fails (interp.R:69-77)
//   4. GLS trend with that model (predict(BLUE=TRUE)): residuals at the stations, their sill
//   5. steps 2-3 again on the GLS residuals -> (nugget, psill, range), or (sill, 0, 0) for a pure nugget.
// Two rules of this library that R does not have, both reported as TWXI_ST_SINGULAR (the oracle raises the same):
//   n < 7 neighbours: at n <= 5 the five-coefficient OLS fits exactly and the residuals are rounding noise, at n = 6 one
//   degree of freedom is left;  two neighbours at the same location (H == 0): V of step 4 has two equal rows.
// One CTA per (point, month): the pair distances come from the station-station table, pair lags are kept in shared memory
// (both variograms share pairs, counts and mean distances), lag sums are accumulated in 64-bit fixed point so that the
// result does not depend on the order of the atomics, the n x n covariance matrix of step 4 is factored in packed shared
// memory.  The gstat calls are [EXT] (SURVEY §8c): restated from the published algorithm, parity unpinned.
#include <algorithm>
#include "twxi_internal.cuh"

namespace twxi {

constexpr int VF_THREADS = 256;
constexpr int VF_WARPS = VF_THREADS / 32;
constexpr int VF_MAXBIN = 512;            // 5 km lags up to a cutoff of 2560 km
constexpr double VF_WIDTH = 5.0;          // interp.R:64 width=5
constexpr double VF_GSCALE = 68719476736.0;     // 2^36: fixed-point scale of the squared differences
constexpr double VF_HSCALE = 1073741824.0;      // 2^30: fixed-point scale of the distances

struct VarioArgs {
    StnTable st;
    int npts, k1, single_mth;
    const int32_t* idx;
    const double* dist;
    const int32_t* nn;
    const double* qlst;        // unused by the fit (the point is not part of the neighbourhood); kept for symmetry
    double* vario;             // [npts][12][3]
    int32_t* status;
};

// sums of NV per-thread values over the CTA, in a fixed order; result valid in every thread after the call
template <int NV>
__device__ __forceinline__ void block_sums(double (&v)[NV], double* red /* [VF_WARPS][NV] */, double* out /* [NV] */) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        const double s = warp_sum(v[i]);
        if (lane == 0) red[warp * NV + i] = s;
    }
    __syncthreads();
    if (threadIdx.x < NV) {
        double s = 0.0;
        for (int w = 0; w < VF_WARPS; ++w) s += red[w * NV + threadIdx.x];
        out[threadIdx.x] = s;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = out[i];
}

// 5x5 SPD solve by Cholesky, one thread.  A packed lower triangle (15), b (5) -> x (5).  false: not positive definite
__device__ bool solve5(const double* A, const double* b, double* x) {
    double L[5][5];
    for (int i = 0; i < 5; ++i)
        for (int j = 0; j <= i; ++j) {
            double s = A[i * (i + 1) / 2 + j];
            for (int k = 0; k < j; ++k) s -= L[i][k] * L[j][k];
            if (i == j) {
                if (!(s > 0.0)) return false;
                L[i][i] = sqrt(s);
            } else {
                L[i][j] = s / L[j][j];
            }
        }
    double y[5];
    for (int i = 0; i < 5; ++i) {
        double s = b[i];
        for (int k = 0; k < i; ++k) s -= L[i][k] * y[k];
        y[i] = s / L[i][i];
    }
    for (int i = 4; i >= 0; --i) {
        double s = y[i];
        for (int k = i + 1; k < 5; ++k) s -= L[k][i] * x[k];
        x[i] = s / L[i][i];
    }
    return true;
}

// Range of the exponential model by weighted least squares (warp 0, all lanes).  bins: bn, bd, bg [K].
// Returns range > 0, or 0 where the R code falls back to the pure nugget.
__device__ double fit_range_warp(int K, const double* bn, const double* bd, const double* bg, double nugget, double psill,
                                 int lane) {
    if (!(psill >= 0.0) || !(nugget >= 0.0) || !isfinite(psill) || !isfinite(nugget)) return 0.0;
    if (nugget == 0.0 && psill == 0.0) return 0.0;
    auto sse = [&](double r) {
        double s = 0.0;
        for (int k = lane; k < K; k += 32) {
            const double h = bd[k];
            const double e = bg[k] - (nugget + psill * (1.0 - exp(-h / r)));
            s += bn[k] / (h * h) * e * e;
        }
        return warp_sum(s);
    };
    double r = 0.1 * bd[K - 1];                               // interp.R:311: 0.10 times the largest lag distance
    if (!(r > 0.0)) return 0.0;
    double s_old = sse(r);
    bool gstat_done = false;
    for (int it = 0; it < 260; ++it) {
        double num = 0.0, den = 0.0;
        for (int k = lane; k < K; k += 32) {
            const double h = bd[k], ex = exp(-h / r), w = bn[k] / (h * h);
            const double e = bg[k] - (nugget + psill * (1.0 - ex));
            const double J = -psill * ex * h / (r * r);       // d model / d range
            num += w * J * e;
            den += w * J * J;
        }
        num = warp_sum(num); den = warp_sum(den);
        if (!(den > 0.0)) return 0.0;                         // singular fit
        double step = num / den, rn = r, s_new = 0.0;
        bool found = false;
        for (int hv = 0; hv < 12; ++hv) {
            rn = r + step;
            if (rn > 0.0) {
                s_new = sse(rn);
                if (s_new <= s_old) { found = true; break; }
            }
            step *= 0.5;
        }
        if (!found) break;
        const bool small_step = fabs(rn - r) <= 1e-10 * rn;
        r = rn;
        // gstat stops when the relative change of the weighted SSE is below 1e-6 (or after 200 iterations); the iteration is
        // continued until the step is below 1e-10 range or no step lowers the SSE, and then polished below
        if (fabs(s_old - s_new) <= 1e-6 * fmax(s_new, 1e-300)) gstat_done = true;
        s_old = s_new;
        if (small_step || (it >= 200 && gstat_done)) break;
    }
    // Within about sqrt(eps) of the minimum the SSE differences above are rounding noise, so the loop stops wherever the
    // noise stops it (1e-10 .. 2e-8 relative).  Newton on the gradient g(r) = sum w J e, whose own rounding is not
    // squared, takes the range to the root of dS/dr: g'(r) = sum w (J' e - J^2) with J' = psill e^(-h/r) h (2r - h) / r^4,
    // a step taken only while S'' > 0 (g' < 0) and |step| <= 1e-3 r, i.e. near a minimum the loop has already reached
    // (where S is nearly flat in r the SSE-tested loop can stop 1e-5 short, so a tighter guard would leave it there).
    for (int it = 0; it < 4 && isfinite(r) && r > 0.0; ++it) {
        double g = 0.0, gp = 0.0;
        for (int k = lane; k < K; k += 32) {
            const double h = bd[k], ex = exp(-h / r), w = bn[k] / (h * h);
            const double e = bg[k] - (nugget + psill * (1.0 - ex));
            const double J = -psill * ex * h / (r * r);
            const double dJ = psill * ex * h * (2.0 * r - h) / (r * r * r * r);
            g += w * J * e;
            gp += w * (dJ * e - J * J);
        }
        g = warp_sum(g); gp = warp_sum(gp);
        if (!(gp < 0.0)) break;
        const double step = -g / gp;
        if (!(fabs(step) <= 1e-3 * r)) break;
        r += step;
    }
    return (isfinite(r) && r > 0.0) ? r : 0.0;
}

__global__ void __launch_bounds__(VF_THREADS) vario_fit_kernel(VarioArgs a, int nmaxv) {
    extern __shared__ __align__(16) double sm[];
    // layout (doubles): X 5 x nmaxv | y | z (residuals) | Z 6 x nmaxv | red 8 x 21 | tot 21 | beta 5 | scal 8 |
    //                   bn, bd, bg VF_MAXBIN each | V packed nmaxv (nmaxv + 1) / 2 | then u64 sg[VF_MAXBIN], int cnt, u16 lag
    double* X = sm;
    double* y = X + 5 * nmaxv;
    double* z = y + nmaxv;
    double* Z = z + nmaxv;
    double* red = Z + 6 * nmaxv;
    double* tot = red + VF_WARPS * 21;
    double* beta = tot + 21;
    double* scal = beta + 5;                                  // 0 sill, 1 nugget, 2 psill, 3 range, 4 ok flag
    double* bn = scal + 8;
    double* bd = bn + VF_MAXBIN;
    double* bg = bd + VF_MAXBIN;
    double* V = bg + VF_MAXBIN;
    unsigned long long* sg = reinterpret_cast<unsigned long long*>(V + (size_t)nmaxv * (nmaxv + 1) / 2);
    unsigned long long* sh = sg + VF_MAXBIN;
    int* cnt = reinterpret_cast<int*>(sh + VF_MAXBIN);
    int* hp = cnt + VF_MAXBIN;
    int* binof = hp + nmaxv;                                  // [VF_MAXBIN] lag -> compact index
    unsigned short* lag = reinterpret_cast<unsigned short*>(binof + VF_MAXBIN);      // [n (n - 1) / 2]
    __shared__ int s_K, s_fail;

    const int nm = a.single_mth >= 0 ? 1 : 12;
    const int q = blockIdx.x / nm;
    const int m = a.single_mth >= 0 ? a.single_mth : blockIdx.x % nm;
    if (a.status[q] != TWXI_ST_OK) return;
    const int n = a.nn[(size_t)q * 24 + m];
    if (n < 1) return;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (n > nmaxv || n < 7) {
        if (tid == 0) atomicCAS(a.status + q, TWXI_ST_OK, n > nmaxv ? TWXI_ST_LIMIT : TWXI_ST_SINGULAR);
        return;
    }
    const int N = a.st.n;
    const int32_t* idx = a.idx + (size_t)q * a.k1;
    const double cutoff = a.dist[(size_t)q * a.k1 + n - 1] * 1.4;      // interp.R:63 (neighbours are in distance order)
    const int nb = (int)floor(cutoff / VF_WIDTH) + 1;
    if (nb > VF_MAXBIN) {
        if (tid == 0) atomicCAS(a.status + q, TWXI_ST_OK, TWXI_ST_LIMIT);
        return;
    }
    if (tid == 0) s_fail = 0;
    // ---- 1. neighbourhood: predictors centred on the nearest neighbour (exact reparametrisation, intercept in X) ----
    const double* lstm = a.st.lst + (size_t)m * N;
    const double* normm = a.st.norm + (size_t)m * N;
    const int s0 = idx[0];
    const double lon0 = a.st.lon[s0], lat0 = a.st.lat[s0], elev0 = a.st.elev[s0], lst0 = lstm[s0];
    for (int j = tid; j < n; j += VF_THREADS) {
        const int s = idx[j];
        hp[j] = a.st.hpos[s];
        X[j] = 1.0;
        X[nmaxv + j] = a.st.lon[s] - lon0;
        X[2 * nmaxv + j] = a.st.lat[s] - lat0;
        X[3 * nmaxv + j] = (a.st.elev[s] - elev0) * 1e-3;
        X[4 * nmaxv + j] = (lstm[s] - lst0) * 0.1;
        y[j] = normm[s];
    }
    for (int b = tid; b < VF_MAXBIN; b += VF_THREADS) { cnt[b] = 0; sh[b] = 0ull; sg[b] = 0ull; }
    __syncthreads();

    // normal equations of [X | rhs] -> beta; used for OLS (X, y) and for GLS (Z = L^-1 [X | y])
    auto normal_solve = [&](const double* Xm, const double* rhs) -> bool {
        double v[21];
#pragma unroll
        for (int i = 0; i < 21; ++i) v[i] = 0.0;
        for (int j = tid; j < n; j += VF_THREADS) {
            double x[5];
#pragma unroll
            for (int c = 0; c < 5; ++c) x[c] = Xm[c * nmaxv + j];
            int t = 0;
#pragma unroll
            for (int i = 0; i < 5; ++i)
#pragma unroll
                for (int c = 0; c <= i; ++c) v[t++] += x[i] * x[c];
#pragma unroll
            for (int i = 0; i < 5; ++i) v[15 + i] += x[i] * rhs[j];
        }
        block_sums<21>(v, red, tot);
        if (tid == 0) {
            double bt[5];
            const bool ok = solve5(tot, tot + 15, bt);
            for (int i = 0; i < 5; ++i) beta[i] = ok ? bt[i] : 0.0;
            scal[4] = ok ? 1.0 : 0.0;
        }
        __syncthreads();
        return scal[4] != 0.0;
    };
    // residuals z = y - X beta, their variance (n - 1) -> scal[0]
    auto residuals = [&]() {
        double v[1] = {0.0};
        for (int j = tid; j < n; j += VF_THREADS) {
            double f = 0.0;
#pragma unroll
            for (int c = 0; c < 5; ++c) f += X[c * nmaxv + j] * beta[c];
            z[j] = y[j] - f;
            v[0] += z[j];
        }
        block_sums<1>(v, red, tot);
        const double mean = v[0] / n;
        double w[1] = {0.0};
        for (int j = tid; j < n; j += VF_THREADS) { const double d = z[j] - mean; w[0] += d * d; }
        block_sums<1>(w, red, tot);
        if (tid == 0) scal[0] = w[0] / (n - 1);
        __syncthreads();
    };
    // gamma sums of the residuals z over the stored pair lags, then compact lags: bn, bd, bg; K -> s_K
    auto variogram = [&](bool first) {
        for (int i = 1 + warp; i < n; i += VF_WARPS) {
            const size_t rowH = (size_t)hp[i] * N;
            const int base = i * (i - 1) / 2;
            for (int j = lane; j < i; j += 32) {
                int b;
                if (first) {
                    const double h = a.st.H[rowH + hp[j]];
                    V[(size_t)i * (i + 1) / 2 + j] = h;       // raw distance, turned into a covariance by the GLS step
                    b = h <= cutoff ? (int)floor(h / VF_WIDTH) : 0xffff;
                    lag[base + j] = (unsigned short)b;
                    if (h == 0.0) s_fail = 1;                 // two neighbours at one location: see the check below
                    if (b != 0xffff) {
                        atomicAdd(&cnt[b], 1);
                        atomicAdd(&sh[b], (unsigned long long)(h * VF_HSCALE + 0.5));
                    }
                } else {
                    b = lag[base + j];
                }
                if (b != 0xffff) {
                    const double d = z[i] - z[j];
                    atomicAdd(&sg[b], (unsigned long long)(d * d * VF_GSCALE + 0.5));
                }
            }
        }
        __syncthreads();
        if (tid == 0) {
            int K = 0;
            double gmin = 1e300;
            for (int b = 0; b < nb; ++b) {
                if (cnt[b] > 0) {
                    bn[K] = (double)cnt[b];
                    bd[K] = (double)sh[b] / VF_HSCALE / cnt[b];
                    bg[K] = (double)sg[b] / VF_GSCALE / (2.0 * cnt[b]);
                    gmin = fmin(gmin, bg[K]);
                    ++K;
                }
                sg[b] = 0ull;
            }
            s_K = K;
            scal[1] = gmin;                                   // nugget fixed at min(gamma), interp.R:68
        }
        __syncthreads();
    };
    // exponential fit -> scal[1..3] = nugget, psill, range (range 0: pure nugget with sill scal[0])
    auto fit = [&]() {
        if (warp == 0) {
            const int K = s_K;
            double rng = 0.0;
            const double nug = scal[1], psill = scal[0] - scal[1];
            if (K > 0) rng = fit_range_warp(K, bn, bd, bg, nug, psill, lane);
            if (lane == 0) { scal[2] = psill; scal[3] = rng; }
        }
        __syncthreads();
    };

    // ---- 2-3. OLS residuals, their variogram, first fit --------------------------------------------------------------
    if (!normal_solve(X, y)) {
        if (tid == 0) atomicCAS(a.status + q, TWXI_ST_OK, TWXI_ST_SINGULAR);
        return;
    }
    residuals();
    variogram(true);
    // two neighbours at the same location make the covariance matrix of step 4 singular (gstat puts nugget + psill at
    // h = 0, so their rows are equal; R stops with an error): decided exactly, as the kriging kernel decides it, instead of
    // by the sign of a rounded pivot, and for a pure nugget too
    if (s_fail) {
        if (tid == 0) atomicCAS(a.status + q, TWXI_ST_OK, TWXI_ST_SINGULAR);
        return;
    }
    fit();

    // ---- 4. GLS trend with the fitted model: beta = (X'V^-1X)^-1 X'V^-1 y -------------------------------------------
    if (scal[3] > 0.0) {
        const double nug = scal[1], psill = scal[2], rinv = -1.0 / scal[3];
        for (int i = warp; i < n; i += VF_WARPS) {
            const size_t base = (size_t)i * (i + 1) / 2;
            for (int j = lane; j <= i; j += 32) V[base + j] = j == i ? nug + psill : psill * exp(V[base + j] * rinv);
        }
        __syncthreads();
        // packed right-looking Cholesky
        for (int k = 0; k < n; ++k) {
            const size_t kk = (size_t)k * (k + 1) / 2 + k;
            if (tid == 0) {
                const double d = V[kk];
                if (!(d > 0.0)) s_fail = 1;
                V[kk] = sqrt(d);
            }
            __syncthreads();
            if (s_fail) break;
            const double piv = V[kk];
            for (int i = k + 1 + tid; i < n; i += VF_THREADS) V[(size_t)i * (i + 1) / 2 + k] /= piv;
            __syncthreads();
            for (int i = k + 1 + warp; i < n; i += VF_WARPS) {
                const size_t base = (size_t)i * (i + 1) / 2;
                const double lik = V[base + k];
                for (int j = k + 1 + lane; j <= i; j += 32) V[base + j] -= lik * V[(size_t)j * (j + 1) / 2 + k];
            }
            __syncthreads();
        }
        if (s_fail) {                                         // covariance matrix not positive definite: R stops with an error
            if (tid == 0) atomicCAS(a.status + q, TWXI_ST_OK, TWXI_ST_SINGULAR);
            return;
        }
        // forward substitution L Z = [X | y]: one warp per right-hand side
        if (warp < 6) {
            const double* rhs = warp < 5 ? X + warp * nmaxv : y;
            double* zc = Z + warp * nmaxv;
            for (int i = 0; i < n; ++i) {
                const size_t base = (size_t)i * (i + 1) / 2;
                double s = 0.0;
                for (int j = lane; j < i; j += 32) s += V[base + j] * zc[j];
                s = warp_sum(s);
                if (lane == 0) zc[i] = (rhs[i] - s) / V[base + i];
                __syncwarp();
            }
        }
        __syncthreads();
        if (!normal_solve(Z, Z + 5 * nmaxv)) {
            if (tid == 0) atomicCAS(a.status + q, TWXI_ST_OK, TWXI_ST_SINGULAR);
            return;
        }
    }
    // ---- 5. GLS residuals (OLS residuals for a pure nugget), second variogram and fit ----------------------------------
    residuals();
    variogram(false);
    fit();
    if (tid == 0) {
        double* o = a.vario + ((size_t)q * 12 + m) * 3;
        if (scal[3] > 0.0) { o[0] = scal[1]; o[1] = scal[2]; o[2] = scal[3]; }
        else { o[0] = scal[0]; o[1] = 0.0; o[2] = 0.0; }      // interp.R:103-107: pure nugget (sill, 0, 0)
    }
}

static size_t vario_smem(int nmaxv) {
    size_t d = (size_t)5 * nmaxv + nmaxv + nmaxv + 6 * nmaxv + VF_WARPS * 21 + 21 + 5 + 8 + 3 * VF_MAXBIN
               + (size_t)nmaxv * (nmaxv + 1) / 2;
    size_t bytes = d * 8 + 2 * VF_MAXBIN * 8 + VF_MAXBIN * 4 + (size_t)nmaxv * 4 + VF_MAXBIN * 4
                   + (size_t)nmaxv * (nmaxv - 1) / 2 * 2 + 16;
    return (bytes + 15) & ~(size_t)15;
}

// Fills b.vario for the (point, month) pairs with nn > 0 (k_norm set by launch_nngh_params or by an override).
int launch_vario_fit(Ctx& c, Batch& b, int mth) {
    if (b.npts <= 0) return TWXI_OK;
    const int nmaxv = std::min(b.k1 - 1, TWXI_MAX_KRIG_NNGHS);
    const size_t smem = vario_smem(nmaxv);
    if (smem > 227 * 1024) { set_error("neighbour count too large for the variogram kernel"); return TWXI_ERR_LIMIT; }
    TWXI_CUDA(cudaFuncSetAttribute(vario_fit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    VarioArgs a;
    a.st = c.st; a.npts = b.npts; a.k1 = b.k1; a.single_mth = mth >= 1 ? mth - 1 : -1;
    a.idx = b.idx; a.dist = b.dist; a.nn = b.nn; a.qlst = b.lst; a.vario = b.vario; a.status = b.status;
    const long long blocks = (long long)b.npts * (mth >= 1 ? 1 : 12);
    vario_fit_kernel<<<(unsigned)blocks, VF_THREADS, smem, c.stream>>>(a, nmaxv);
    TWXI_LAUNCH_CHECK();
    return TWXI_OK;
}

}  // namespace twxi

// C ABI of maxent_b200 (include/maxent_b200.h) + the small kernels around the alpha sweep:
// V' re-tiling, TauKernel and IOmegaKernel fills, data projection, analyzer reductions.
#include <stdlib.h>
#include "mx_common.cuh"
#include <stdio.h>
#include <stdint.h>

namespace mx {


// ---- V' [n_omega, s] row-major -> [n_kt][NT][64] swizzled tiles (zero padded) ---------------------
__global__ void layout_V_kernel(const double* __restrict__ V, int n_omega, int s, int NT, double* __restrict__ Vt, int64_t total) {
    for (int64_t o = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; o < total; o += (int64_t)gridDim.x * blockDim.x) {
        const int64_t tile = o / 64;
        const int e64 = (int)(o - tile * 64);
        const int kt = (int)(tile / NT), jt = (int)(tile - (int64_t)kt * NT);
        // invert tile_off by search (64 candidates; runs once per problem)
        int n = 0, c = 0;
        for (int nn = 0; nn < 8; ++nn)
            for (int cc = 0; cc < 8; ++cc)
                if (tile_off(nn, cc) == e64) { n = nn; c = cc; }
        const int k = kt * 8 + n, j = jt * 8 + c;
        Vt[o] = (k < n_omega && j < s) ? V[(int64_t)k * s + j] : 0.0;
    }
}

// ---- TauKernel._fill_values (python/kernels.py:253-263) --------------------------------------------------
__global__ void tau_kernel_kernel(const double* __restrict__ tau, const double* __restrict__ omega,
                                  int n_tau, int n_omega, double beta, double* __restrict__ K) {
    const int64_t total = (int64_t)n_tau * n_omega;
    for (int64_t o = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; o < total; o += (int64_t)gridDim.x * blockDim.x) {
        const int i = (int)(o / n_omega), j = (int)(o - (int64_t)i * n_omega);
        const double w = omega[j], t = tau[i];
        double v;
        if (w >= 0.0) v = -exp(-w * t) / (exp(-beta * w) + 1.0);
        else          v = -exp(w * (beta - t)) / (1.0 + exp(beta * w));
        K[o] = v;
    }
}

// ---- IOmegaKernel.fused_matrix (python/kernels.py:283-346): K[2 n_iw, n_omega] = [Re; Im] 1 / (i nu_n - omega) ----
// Evaluated as numpy divides complex numbers (Smith's algorithm on 1 / (-omega + i nu), no contracted products), so that
// the device fill reproduces the host matrix of IOmegaKernel to the last bits.
__global__ void iomega_kernel_kernel(const double* __restrict__ iomega, const double* __restrict__ omega,
                                     int n_iw, int n_omega, double* __restrict__ K) {
    const int64_t total = (int64_t)n_iw * n_omega;
    for (int64_t o = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; o < total; o += (int64_t)gridDim.x * blockDim.x) {
        const int i = (int)(o / n_omega), j = (int)(o - (int64_t)i * n_omega);
        const double br = -omega[j], bi = iomega[i];         // denominator br + i bi
        double re, im;
        if (fabs(br) >= fabs(bi)) {
            if (br == 0.0 && bi == 0.0) { re = 1.0 / fabs(br); im = 0.0 / fabs(br); }
            else {
                const double rat = bi / br, scl = 1.0 / __dadd_rn(br, __dmul_rn(bi, rat));
                re = __dmul_rn(__dadd_rn(1.0, __dmul_rn(0.0, rat)), scl);
                im = __dmul_rn(__dsub_rn(0.0, rat), scl);
            }
        } else {
            const double rat = br / bi, scl = 1.0 / __dadd_rn(bi, __dmul_rn(br, rat));
            re = __dmul_rn(__dadd_rn(rat, 0.0), scl);
            im = __dmul_rn(__dsub_rn(__dmul_rn(0.0, rat), 1.0), scl);
        }
        K[o] = re;
        K[o + total] = im;
    }
}

// ---- data projection: gt = Qw^T G ; c0 = |sqrtw*G - Qo gt|^2   (one CTA per spectrum) -----------------
__global__ void __launch_bounds__(256) project_kernel(const double* __restrict__ Qw, const double* __restrict__ Qo,
                                                      const double* __restrict__ sqrtw, const double* __restrict__ G,
                                                      int n_tau, int s, double* __restrict__ gt, double* __restrict__ c0) {
    __shared__ double sg[MX_MAX_NSV];
    __shared__ double red[8];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double* Gb = G + (int64_t)b * n_tau;
    for (int j = warp; j < s; j += 8) {
        double acc = 0.0;
        for (int i = lane; i < n_tau; i += 32) acc = fma(Qw[(int64_t)i * s + j], Gb[i], acc);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) { sg[j] = acc; gt[(int64_t)b * s + j] = acc; }
    }
    __syncthreads();
    double part = 0.0;
    for (int i = tid; i < n_tau; i += 256) {
        double r = sqrtw[i] * Gb[i];
        const double* q = Qo + (int64_t)i * s;
        for (int j = 0; j < s; ++j) r = fma(-q[j], sg[j], r);
        part = fma(r, r, part);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if (lane == 0) red[warp] = part;
    __syncthreads();
    if (tid == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += red[w];
        c0[b] = t;
    }
}

// ---- analyzers (python/analyzers/*.py), one warp-sized CTA per spectrum; n_alpha <= 1024 ----------------
// Line fits are done in closed form on centred sums (np.polyfit solves the same least squares).
__device__ double line_resid(const double* x, const double* y, int i0, int i1, int deg, double* slope, double* icpt) {
    // least squares over indices [i0, i1) skipping NaN y; returns the residual sum of squares
    int n = 0; double mx = 0, my = 0;
    for (int i = i0; i < i1; ++i) if (!isnan(y[i])) { mx += x[i]; my += y[i]; ++n; }
    // np.polyfit raises TypeError on an empty piece and fit_piecewise then excludes this break point
    // (linefit_analyzer.py:62-75): the residual is NaN, not 0
    if (n == 0) { *slope = nan(""); *icpt = nan(""); return nan(""); }
    mx /= n; my /= n;
    double sxx = 0, sxy = 0, syy = 0;
    for (int i = i0; i < i1; ++i) if (!isnan(y[i])) { const double dx = x[i] - mx, dy = y[i] - my; sxx += dx * dx; sxy += dx * dy; syy += dy * dy; }
    if (deg == 0) { *slope = 0.0; *icpt = my; return n > 1 ? syy : 0.0; }
    // one point (or all x equal): np.polyfit returns the minimum-norm line of its column-scaled problem, y / (2x) and y / 2
    if (n < 2 || sxx == 0.0) { *slope = mx != 0.0 ? my / (2.0 * mx) : 0.0; *icpt = mx != 0.0 ? 0.5 * my : my; return 0.0; }
    const double m = sxy / sxx;
    *slope = m; *icpt = my - m * mx;
    double r = 0;
    for (int i = i0; i < i1; ++i) if (!isnan(y[i])) { const double d = (y[i] - my) - m * (x[i] - mx); r += d * d; }
    return n > 2 ? r : 0.0;      // np.polyfit returns no residual when the fit is exact-determined
}

__global__ void __launch_bounds__(128) analyze_kernel(const double* __restrict__ alpha, const double* __restrict__ chi2,
                                                      const double* __restrict__ S, const double* __restrict__ logp,
                                                      const double* __restrict__ A, int n_alpha, int n_omega,
                                                      double gamma, int linefit_deg, int by_integration,
                                                      int* __restrict__ aidx, double* __restrict__ A_out,
                                                      double* __restrict__ aux) {
    extern __shared__ double sh[];
    double* lx = sh;                    // log alpha
    double* ly = lx + n_alpha;          // log chi2
    double* cost = ly + n_alpha;        // piecewise misfit / scratch
    double* wts = cost + n_alpha;       // bryan weights
    __shared__ int idx[MX_N_ANALYZERS];
    const int b = blockIdx.x, tid = threadIdx.x;
    const double* c2 = chi2 + (int64_t)b * n_alpha;
    const double* Sb = S + (int64_t)b * n_alpha;
    const double* pb = logp ? logp + (int64_t)b * n_alpha : nullptr;
    // aux row: [0..3] line-fit parameters (slope, intercept of both pieces), then curvature[n_alpha], dS/dlog(alpha)[n_alpha]
    double* ax = aux ? aux + (int64_t)b * (4 + 2 * n_alpha) : nullptr;
    if (ax) for (int i = tid; i < 4 + 2 * n_alpha; i += blockDim.x) ax[i] = nan("");
    for (int i = tid; i < n_alpha; i += blockDim.x) { lx[i] = log(alpha[i]); ly[i] = log(c2[i]); cost[i] = nan(""); }
    if (tid < MX_N_ANALYZERS) idx[tid] = -1;
    __syncthreads();
    // --- LineFit: fit_piecewise (linefit_analyzer.py:28-87) ---
    double* p1s = wts;  // reuse as scratch before the Bryan weights are formed
    for (int i = 2 + tid; i < n_alpha - 2; i += blockDim.x) {
        double m1, c1, m2, c2_;
        const double r1 = line_resid(lx, ly, 0, i, 1, &m1, &c1);
        const double r2 = line_resid(lx, ly, i, n_alpha, linefit_deg, &m2, &c2_);
        cost[i] = r1 + r2;
    }
    __syncthreads();
    if (tid == 0) {
        int best = -1; double bv = 0;
        for (int i = 0; i < n_alpha; ++i) if (!isnan(cost[i]) && (best < 0 || cost[i] < bv)) { best = i; bv = cost[i]; }
        if (best >= 0) {
            double m1, c1, m2, c2_;
            line_resid(lx, ly, 0, best, 1, &m1, &c1);
            line_resid(lx, ly, best, n_alpha, linefit_deg, &m2, &c2_);
            const double X = (c2_ - c1) / (m1 - (linefit_deg == 1 ? m2 : 0.0));
            int k = -1; double kv = 0;
            for (int i = 0; i < n_alpha; ++i) { const double d = fabs(lx[i] - X); if (!isnan(d) && (k < 0 || d < kv)) { k = i; kv = d; } }
            idx[MX_AN_LINEFIT] = k;
            if (ax) { ax[0] = m1; ax[1] = c1; ax[2] = (linefit_deg == 1 ? m2 : 0.0); ax[3] = c2_; }
        }
        (void)p1s;
    }
    // --- Chi2Curvature (chi2_curvature_analyzer.py:25-49,120-122): x = gamma log10 alpha, y = log10 chi2 ---
    if (tid == 32) {
        const double il10 = 1.0 / log(10.0);
        int k = -1; double kv = 0;
        for (int i = 1; i < n_alpha - 1; ++i) {
            const double x0 = gamma * log10(alpha[i - 1]), x1 = gamma * log10(alpha[i]), x2 = gamma * log10(alpha[i + 1]);
            const double y0 = log10(c2[i - 1]), y1 = log10(c2[i]), y2 = log10(c2[i + 1]);
            const double d2 = (y2 - 2 * y1 + y0) / ((x2 - x1) * (x1 - x0));
            const double d1 = ((y2 - y1) / (x2 - x1) + (y1 - y0) / (x1 - x0)) / 2;
            const double cv = d2 / pow(1 + d1 * d1, 1.5);
            if (ax) ax[4 + i] = cv;
            if (!isnan(cv) && (k < 0 || cv > kv)) { k = i; kv = cv; }
        }
        (void)il10;
        idx[MX_AN_CHI2CURV] = k;
    }
    // --- Entropy (entropy_analyzer.py:92-95) ---
    if (tid == 64) {
        int k = -1; double kv = 0;
        for (int i = 1; i < n_alpha - 1; ++i) {
            const double d = (Sb[i + 1] - Sb[i - 1]) / (log(alpha[i + 1]) - log(alpha[i - 1]));
            const double v = d * d;
            if (ax) ax[4 + n_alpha + i] = d;
            if (!isnan(v) && (k < 0 || v < kv)) { k = i; kv = v; }
        }
        idx[MX_AN_ENTROPY] = k;
    }
    // --- Classic (classic_analyzer.py:70-76) ---
    if (tid == 96 && pb) {
        int k = -1; double kv = 0;
        for (int i = 0; i < n_alpha; ++i) if (!isnan(pb[i]) && (k < 0 || pb[i] > kv)) { k = i; kv = pb[i]; }
        idx[MX_AN_CLASSIC] = k;
    }
    __syncthreads();
    // --- Bryan weights (bryan_analyzer.py:133-143) ---
    __shared__ int have_p;
    if (tid == 0) {
        have_p = 0;
        if (pb) {
            double mxp = 0; int any = 0;
            for (int i = 0; i < n_alpha; ++i) if (!isnan(pb[i]) && (!any || pb[i] > mxp)) { mxp = pb[i]; any = 1; }
            if (any) {
                have_p = 1;
                for (int i = 0; i < n_alpha; ++i) wts[i] = exp(pb[i] - mxp);
                double norm = 0;
                if (by_integration) {
                    // trapz over the non-NaN subset, then multiply by trapezoid weights of that subset
                    int prev = -1;
                    for (int i = 0; i < n_alpha; ++i) if (!isnan(wts[i])) { if (prev >= 0) norm += 0.5 * (wts[i] + wts[prev]) * (alpha[i] - alpha[prev]); prev = i; }
                    int pprev = -1; prev = -1;
                    // delta_alpha on the subset
                    for (int i = 0; i < n_alpha; ++i) cost[i] = nan("");
                    int first = -1, last = -1;
                    for (int i = 0; i < n_alpha; ++i) if (!isnan(wts[i])) { if (first < 0) first = i; last = i; }
                    prev = -1;
                    for (int i = 0; i < n_alpha; ++i) if (!isnan(wts[i])) {
                        int nxt = -1; for (int k = i + 1; k < n_alpha; ++k) if (!isnan(wts[k])) { nxt = k; break; }
                        double d;
                        if (prev < 0 && nxt >= 0) d = (alpha[nxt] - alpha[i]) / 2.0;
                        else if (nxt < 0 && prev >= 0) d = (alpha[i] - alpha[prev]) / 2.0;
                        else if (prev >= 0 && nxt >= 0) d = (alpha[nxt] - alpha[prev]) / 2.0;
                        else d = nan("");
                        cost[i] = d; prev = i;
                    }
                    (void)pprev;
                    for (int i = 0; i < n_alpha; ++i) if (!isnan(wts[i])) wts[i] = wts[i] / norm * cost[i];
                } else {
                    for (int i = 0; i < n_alpha; ++i) if (!isnan(wts[i])) norm += wts[i];
                    for (int i = 0; i < n_alpha; ++i) if (!isnan(wts[i])) wts[i] /= norm;
                }
                idx[MX_AN_BRYAN] = 0;   // "available"
            }
        }
    }
    __syncthreads();
    if (tid < MX_N_ANALYZERS) aidx[(int64_t)b * MX_N_ANALYZERS + tid] = idx[tid];
    if (A_out == nullptr || A == nullptr) return;
    const double* Ab = A + (int64_t)b * n_alpha * n_omega;
    double* Ob = A_out + (int64_t)b * MX_N_ANALYZERS * n_omega;
    for (int k = tid; k < n_omega; k += blockDim.x) {
        for (int an = 0; an < 4; ++an) Ob[(int64_t)an * n_omega + k] = idx[an] >= 0 ? Ab[(int64_t)idx[an] * n_omega + k] : nan("");
        double acc = nan("");
        if (have_p) {
            acc = 0.0;
            for (int i = 0; i < n_alpha; ++i) if (!isnan(wts[i])) acc += wts[i] * Ab[(int64_t)i * n_omega + k];
        }
        Ob[(int64_t)MX_AN_BRYAN * n_omega + k] = acc;
    }
}

// ---- PoormanMaxEnt off-diagonal default models (python/elementwise_maxent.py:633-652), one CTA per spectrum p -------
// D[p] = (sqrt(A_i A_j) + d_add) * delta from the diagonal pass's analyzer output, and the initial vector
// v0[p] = V'_g^T log(arg(H0, D[p])) of the plus-minus entropy (engine.per_spectrum_models).  v0 is summed over omega in
// index order by one thread per singular component, so every spectrum's result is independent of P and of its position.
__global__ void __launch_bounds__(256) poorman_models_kernel(const double* __restrict__ A_out, int slot,
                                                             const int32_t* __restrict__ rows,
                                                             const double* __restrict__ delta, double d_add,
                                                             const double* __restrict__ A_init,
                                                             const double* __restrict__ Vp,
                                                             const int32_t* __restrict__ group, int n_omega, int n_sv,
                                                             int ldD, double* __restrict__ D, double* __restrict__ v0,
                                                             int32_t* __restrict__ ok) {
    extern __shared__ double larg[];    // log(arg) of this spectrum, [n_omega]
    const int p = blockIdx.x, tid = threadIdx.x;
    const double* Ai = A_out + ((int64_t)rows[2 * p] * MX_N_ANALYZERS + slot) * n_omega;
    const double* Aj = A_out + ((int64_t)rows[2 * p + 1] * MX_N_ANALYZERS + slot) * n_omega;
    double* Dp = D + (int64_t)p * ldD;
    int nan_seen = 0;
    for (int w = tid; w < n_omega; w += blockDim.x) {
        const double ai = Ai[w], aj = Aj[w];
        nan_seen |= isnan(ai) || isnan(aj);
        // explicit rounding steps: the same operations, in the same order, as DataDefaultModel(np.sqrt(.) + c).D
        const double Dw = __dmul_rn(__dadd_rn(__dsqrt_rn(__dmul_rn(ai, aj)), d_add), delta[w]);
        Dp[w] = Dw;
        const double H0 = (A_init ? A_init[w] : Dw) * delta[w];      // maxent_loop.py:196-203 quirk
        double arg = (H0 + sqrt(H0 * H0 + 4.0 * Dw * Dw)) / (2.0 * Dw);   // functions.py:793-796
        if (fabs(arg) <= 1e-100) arg = 1e-100;
        larg[w] = log(arg);
    }
    for (int w = n_omega + tid; w < ldD; w += blockDim.x) Dp[w] = 0.0;
    const int any_nan = __syncthreads_or(nan_seen);
    if (tid == 0) ok[p] = any_nan ? 0 : 1;
    const double* V = Vp + (group ? (int64_t)group[p] * n_omega * n_sv : 0);
    for (int k = tid; k < n_sv; k += blockDim.x) {
        double acc = 0.0;
        for (int w = 0; w < n_omega; ++w) acc = fma(V[(int64_t)w * n_sv + k], larg[w], acc);
        v0[(int64_t)p * n_sv + k] = acc;
    }
}

// ---- measurement helper: FP64 pipe peak (the roofline denominator of the sweep kernel) --------------------------
// Every SM runs 2 x 8 warps of independent DMMA (m8n8k4) or DFMA chains: what the FP64 pipe delivers when nothing else
// limits it.  bench.py calls this inside the benchmark run (MEASURED_PEAKS.json carries no FP64 figure).
template <bool MMA>
__global__ void __launch_bounds__(256) fp64_peak_kernel(double* out, double a, double b, int iters) {
    double c[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) c[i] = threadIdx.x * 1e-3 + i;
    for (int it = 0; it < iters; ++it) {
        if (MMA) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                double acc[2] = {c[2 * i], c[2 * i + 1]};
                dmma(acc, a, b);
                c[2 * i] = acc[0]; c[2 * i + 1] = acc[1];
            }
        } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) c[i] = fma(c[i], a, b);
        }
    }
    double s = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += c[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

}  // namespace mx

using namespace mx;

extern "C" {

const char* mx_version(void) { return "maxent_b200 0.1 (sm_100a)"; }

int mx_device_sm_count(void) {
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return MX_ERR_NO_DEVICE;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return MX_ERR_NO_DEVICE;
    return sms;
}

int64_t mx_layout_V_size(int32_t n_omega, int32_t n_sv) {
    if (n_omega < 1 || n_sv < 1 || n_sv > MX_MAX_NSV) return MX_ERR_BAD_ARG;
    const int64_t n_kt = (n_omega + 7) / 8;
    return n_kt * sweep_tiles(n_sv) * 64;
}

int mx_layout_V(const double* V, int32_t n_omega, int32_t n_sv, double* Vt, void* stream) {
    const int64_t total = mx_layout_V_size(n_omega, n_sv);
    if (total < 0 || !V || !Vt) return MX_ERR_BAD_ARG;
    const int nt = sweep_tiles(n_sv);
    const int grid = (int)((total + 255) / 256 < 1184 ? (total + 255) / 256 : 1184);
    layout_V_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(V, n_omega, n_sv, nt, Vt, total);
    return cudaGetLastError() == cudaSuccess ? MX_OK : MX_ERR_CUDA;
}

int mx_tau_kernel(const double* tau, const double* omega, int32_t n_tau, int32_t n_omega, double beta,
                  double* K, void* stream) {
    if (!tau || !omega || !K || n_tau < 1 || n_omega < 1) return MX_ERR_BAD_ARG;
    const int64_t total = (int64_t)n_tau * n_omega;
    const int grid = (int)((total + 255) / 256 < 1184 ? (total + 255) / 256 : 1184);
    tau_kernel_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(tau, omega, n_tau, n_omega, beta, K);
    return cudaGetLastError() == cudaSuccess ? MX_OK : MX_ERR_CUDA;
}

int mx_iomega_kernel(const double* iomega, const double* omega, int32_t n_iw, int32_t n_omega, double* K, void* stream) {
    if (!iomega || !omega || !K || n_iw < 1 || n_omega < 1) return MX_ERR_BAD_ARG;
    const int64_t total = (int64_t)n_iw * n_omega;
    const int grid = (int)((total + 255) / 256 < 1184 ? (total + 255) / 256 : 1184);
    iomega_kernel_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(iomega, omega, n_iw, n_omega, K);
    return cudaGetLastError() == cudaSuccess ? MX_OK : MX_ERR_CUDA;
}

int mx_svd_jacobi(const double* K, int32_t m, int32_t n, double* U, double* S, double* V, double* work,
                  int32_t max_sweeps, int32_t* sweeps_done, void* stream) {
    if (!K || !U || !S || !V || !work || m < n || n < 1) return MX_ERR_BAD_ARG;
    return svd_jacobi(K, m, n, U, S, V, work, max_sweeps, sweeps_done, (cudaStream_t)stream);
}

int mx_fp64_peak(double* tflops_dmma, double* tflops_dfma, double* scratch, void* stream_) {
    if (!tflops_dmma || !tflops_dfma || !scratch) return MX_ERR_BAD_ARG;
    cudaStream_t stream = (cudaStream_t)stream_;
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return MX_ERR_NO_DEVICE;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaEvent_t e0, e1;
    if (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess) return MX_ERR_CUDA;
    const int grid = 2 * sms, iters = 1 << 15;
    double best[2] = {0.0, 0.0};
    for (int kind = 0; kind < 2; ++kind)
        for (int rep = 0; rep < 4; ++rep) {          // first repetition warms up
            cudaEventRecord(e0, stream);
            if (kind == 0) fp64_peak_kernel<true><<<grid, 256, 0, stream>>>(scratch, 1e-3, 1e-3, iters);
            else fp64_peak_kernel<false><<<grid, 256, 0, stream>>>(scratch, 1.0000001, 1e-9, iters);
            cudaEventRecord(e1, stream);
            if (cudaEventSynchronize(e1) != cudaSuccess) return MX_ERR_CUDA;
            float ms = 0.f;
            cudaEventElapsedTime(&ms, e0, e1);
            // flops per thread and iteration: 8 DMMA x 512 / 32 lanes = 128, or 16 FMA x 2 = 32
            const double fl = (double)grid * 256 * iters * (kind == 0 ? 128.0 : 32.0);
            const double tf = fl / (ms * 1e-3) / 1e12;
            if (rep > 0 && tf > best[kind]) best[kind] = tf;
        }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *tflops_dmma = best[0];
    *tflops_dfma = best[1];
    return cudaGetLastError() == cudaSuccess ? MX_OK : MX_ERR_CUDA;
}

int mx_gram_schmidt_rows(double* Yt, int32_t len, int32_t p, double drop_rel, void* stream) {
    if (!Yt || len < 1 || p < 1 || p > 512) return MX_ERR_BAD_ARG;
    return mx::gram_schmidt_rows(Yt, len, p, drop_rel, (cudaStream_t)stream);
}

int64_t mx_svd_truncated_work_doubles(int32_t m, int32_t n, int32_t p) {
    if (m < 1 || n < 1 || p < 1 || p > m || p > n) return MX_ERR_BAD_ARG;
    return svd_truncated_work_doubles(m, n, p);
}

int mx_svd_truncated(const double* K, int32_t m, int32_t n, int32_t p, double* U, double* S, double* V, double* work,
                     uint64_t seed, void* stream) {
    if (!K || !U || !S || !V || !work || m < 1 || n < 1 || p < 1 || p > m || p > n) return MX_ERR_BAD_ARG;
    return svd_truncated(K, m, n, p, U, S, V, work, seed, (cudaStream_t)stream);
}

int mx_project_data(const MxProblem* p, const double* G, int32_t B, double* gt, double* c0, void* stream) {
    if (B == 0) return MX_OK;
    if (!p || !G || !gt || !c0 || B < 0) return MX_ERR_BAD_ARG;
    if (p->n_sv < 1 || p->n_sv > MX_MAX_NSV) return MX_ERR_UNSUPPORTED;
    project_kernel<<<B, 256, 0, (cudaStream_t)stream>>>(p->Qw, p->Qo, p->sqrtw, G, p->n_tau, p->n_sv, gt, c0);
    return cudaGetLastError() == cudaSuccess ? MX_OK : MX_ERR_CUDA;
}

static int fill_args(const MxProblem* p, SweepArgs& a) {
    if (p->n_sv < 1 || p->n_omega < 1 || p->n_alpha < 1) return MX_ERR_BAD_ARG;
    if (p->variant < 0 || p->variant > 2) return MX_ERR_BAD_ARG;
    if (!(p->lm.nu > 1.0)) return MX_ERR_BAD_ARG;     // levenberg_minimizer.py:139-140
    a.n_omega = p->n_omega; a.n_kt = (p->n_omega + 7) / 8; a.n_sv = p->n_sv; a.n_alpha = p->n_alpha;
    a.variant = p->variant; a.want_prob = p->want_probability; a.pk = 0;
    a.maxiter = p->lm.maxiter; a.miniter = p->lm.miniter;
    a.mu0 = p->lm.mu0; a.nu = p->lm.nu; a.max_mu = p->lm.max_mu;
    a.conv_maxd = p->lm.conv_max_derivative; a.conv_relq = p->lm.conv_rel_change; a.eta = p->chi2_factor;
    a.conv_absq = p->lm.conv_abs_change; a.marquardt = p->lm.marquardt ? 1 : 0;
    a.per_spec = (p->per_spectrum_model & MX_PER_SPECTRUM_MODEL) ? 1 : 0;
    a.per_spec_xi = (p->per_spectrum_model & MX_PER_SPECTRUM_XI) ? 1 : 0;
    a.per_spec_alpha = (p->per_spectrum_model & MX_PER_SPECTRUM_ALPHA) ? 1 : 0;
    a.Vt = p->Vt; a.D = p->D; a.delta = p->delta; a.xi = p->xi; a.alpha = p->alpha; a.v0 = p->v0;
    a.vt_index = (p->per_spectrum_model & MX_PER_SPECTRUM_VT) ? p->vt_index : nullptr;
    a.vt_stride = p->vt_stride;
    if ((p->per_spectrum_model & MX_PER_SPECTRUM_VT) && (!p->vt_index || p->vt_stride < 1)) return MX_ERR_BAD_ARG;
    return MX_OK;
}

int mx_sweep_config(int32_t n_sv, int32_t* smem_bytes, int32_t* threads) {
    SweepArgs a = {};
    a.n_sv = n_sv;
    a.B = 1;
    a.conv_absq = -1.0;
    int sm = 0;
    const int rc = dispatch_sweep(a, nullptr, true, &sm, nullptr);
    if (rc != MX_OK) return rc;
    if (smem_bytes) *smem_bytes = sm;
    if (threads) *threads = sweep_threads();
    return MX_OK;
}

static const int64_t WS_HEADER = 256;     // bytes reserved for the work counter in front of the scratch rows

// fills a for a sweep of B spectra of p and finds the persistent CTAs it would be launched with (what the workspace is
// sized for)
static int sweep_grid(const MxProblem* p, int32_t B, SweepArgs& a, int* grid) {
    int rc = fill_args(p, a);
    if (rc != MX_OK) return rc;
    a.B = B > 0 ? B : 1;
    *grid = 0;
    rc = dispatch_sweep(a, nullptr, true, nullptr, grid);
    if (rc != MX_OK) return rc;
    return *grid > 0 ? MX_OK : MX_ERR_NO_DEVICE;
}

// work counter + scratch rows + wide slices of a sweep of p on `grid` CTAs
static int64_t sweep_workspace_bytes(const MxProblem* p, int grid) {
    return WS_HEADER + 8 * sweep_scratch_doubles(p->n_sv, p->n_omega, p->variant, grid);
}

int64_t mx_sweep_workspace_bytes(const MxProblem* p, int32_t B) {
    if (!p || B < 0) return MX_ERR_BAD_ARG;
    SweepArgs a = {};
    int grid = 0;
    const int rc = sweep_grid(p, B, a, &grid);
    if (rc != MX_OK) return rc;
    return sweep_workspace_bytes(p, grid);
}

int mx_alpha_sweep(const MxProblem* p, const double* gt, const double* c0, int32_t B, const MxSweepOut* out,
                   void* workspace, int64_t workspace_bytes, void* stream) {
    if (B == 0) return MX_OK;
    if (!p || !gt || !c0 || !out || !workspace || B < 0) return MX_ERR_BAD_ARG;
    if (!out->chi2 || !out->S || !out->Q) return MX_ERR_BAD_ARG;
    SweepArgs a = {};
    int grid = 0;
    const int rc = sweep_grid(p, B, a, &grid);
    if (rc != MX_OK) return rc;
    if (workspace_bytes < sweep_workspace_bytes(p, grid) || (reinterpret_cast<uintptr_t>(workspace) & 15) != 0)
        return MX_ERR_BAD_ARG;
    a.gt = gt; a.c0 = c0;
    a.o_v = out->v; a.o_A = out->A; a.o_chi2 = out->chi2; a.o_S = out->S; a.o_Q = out->Q; a.o_logp = out->logp;
    a.o_niter = out->n_iter; a.o_nq = out->n_qeval; a.o_ns = out->n_solve; a.o_status = out->status;
    a.o_ntrial = out->n_trial; a.o_nbatch = out->n_batch; a.o_phase = reinterpret_cast<long long*>(out->phase_cycles);
    a.counter = reinterpret_cast<int*>(workspace);
    a.scratch = reinterpret_cast<double*>(reinterpret_cast<char*>(workspace) + WS_HEADER);
    a.wide_stride = sweep_wide_stride(p->n_sv);         // the slices of the wide instantiations follow the scratch rows
    a.wide = a.wide_stride ? a.scratch + sweep_rows_doubles(p->n_omega, p->variant, grid) : nullptr;
    if (cudaMemsetAsync(workspace, 0, WS_HEADER, (cudaStream_t)stream) != cudaSuccess) return MX_ERR_CUDA;
    return dispatch_sweep(a, (cudaStream_t)stream, false, nullptr, nullptr);
}

int mx_analyze(const double* alpha, const double* chi2, const double* S, const double* logp, const double* A,
               int32_t B, int32_t n_alpha, int32_t n_omega, double gamma, int32_t linefit_deg,
               int32_t bryan_by_integration, int32_t* alpha_index, double* A_out, double* aux, void* stream) {
    if (B == 0) return MX_OK;
    if (!alpha || !chi2 || !S || !alpha_index || B < 0 || n_alpha < 1 || n_alpha > 1024) return MX_ERR_BAD_ARG;
    const size_t shb = 4 * (size_t)n_alpha * sizeof(double);
    analyze_kernel<<<B, 128, shb, (cudaStream_t)stream>>>(alpha, chi2, S, logp, A, n_alpha, n_omega, gamma,
                                                          linefit_deg, bryan_by_integration, alpha_index, A_out, aux);
    return cudaGetLastError() == cudaSuccess ? MX_OK : MX_ERR_CUDA;
}

int mx_poorman_models(const double* A_out, int32_t slot, const int32_t* rows, int32_t P, const double* delta,
                      double d_add, const double* A_init, const double* Vp, const int32_t* group, int32_t n_omega,
                      int32_t n_sv, double* D, double* v0, int32_t* ok, void* stream) {
    if (P == 0) return MX_OK;
    if (!A_out || !rows || !delta || !Vp || !D || !v0 || !ok || P < 0 || slot < 0 || slot >= MX_N_ANALYZERS
        || n_omega < 1 || n_sv < 1 || n_sv > MX_MAX_NSV) return MX_ERR_BAD_ARG;
    const size_t shb = (size_t)n_omega * sizeof(double);
    if (shb > 227 * 1024) return MX_ERR_UNSUPPORTED;
    if (shb > 48 * 1024 &&
        cudaFuncSetAttribute(poorman_models_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shb) != cudaSuccess)
        return MX_ERR_CUDA;
    poorman_models_kernel<<<P, 256, shb, (cudaStream_t)stream>>>(A_out, slot, rows, delta, d_add, A_init, Vp, group,
                                                                 n_omega, n_sv, (n_omega + 1) & ~1, D, v0, ok);
    return cudaGetLastError() == cudaSuccess ? MX_OK : MX_ERR_CUDA;
}

}  // extern "C"

// Retarded transform of spectra on the omega mesh: G_r(z_k) = int dx A_r(x) / (z_k - x), z_k = w_k + i eta, for A_r
// linear between the mesh nodes and zero outside them (the spectrum whose integral the trapezoid weights give).
// The transform is linear in A: G_r(z_k) = sum_j M[k, j] A_rj with a complex table M that depends on (mesh, w, eta)
// only (mx_hilbert_table); mx_hilbert_apply is the product A M^T for many spectra on the FP64 tensor cores, with the
// self-energy algebra of the continuators in its epilogue.
#include "mx_common.cuh"

namespace mx {

namespace {

struct cplx {
    double re, im;
};
__device__ __forceinline__ cplx cmul(cplx a, cplx b) { return {a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re}; }
__device__ __forceinline__ cplx cadd(cplx a, cplx b) { return {a.re + b.re, a.im + b.im}; }

// Coefficients of A_a and A_b in the integral over one segment [x_a, x_b] (h = x_b - x_a), written in
// q = (z - x_b) / h and L = log((z - x_a) / (z - x_b)) = log(1 + 1/q):
//     int = (A_a + s (z - x_a)) L - (A_b - A_a),  s = (A_b - A_a) / h
//   => c_a = 1 - q L,  c_b = (q + 1) L - 1.
// Far from the segment (|q| > 10, i.e. h << |z - x_b|) L = log1p(t), t = 1/q, is close to t and both coefficients are
// O(t) differences of O(1) terms, which would lose the digits of 1/|t|; there they come from the series of log1p
// with the cancellation done exactly: c_a = sum_n (-1)^(n+1) t^n / (n+1), c_b = sum_n (-1)^(n+1) t^n / (n (n+1)),
// truncated where |t|^n < 1e-17.  Near it, L = log(|u| / |q|) + i (arg u - arg q) with u = q + 1 = (z - x_a) / h;
// both arguments lie in (0, pi) for Im z > 0, so their difference is the principal branch of the ratio's log.
constexpr double HB_FAR_Q = 10.0;
constexpr int HB_SERIES_TERMS = 18;

__device__ void segment_coeffs(double x_a, double x_b, double w, double eta, cplx* c_a, cplx* c_b) {
    const double h = x_b - x_a;
    const cplx q = {(w - x_b) / h, eta / h};
    const double q2 = q.re * q.re + q.im * q.im;
    if (q2 > HB_FAR_Q * HB_FAR_Q) {
        const cplx t = {q.re / q2, -q.im / q2};
        cplx sa = {0.0, 0.0}, sb = {0.0, 0.0};
        for (int n = HB_SERIES_TERMS; n >= 1; --n) {       // Horner: s = t (a_n + s)
            const double sgn = (n & 1) ? 1.0 : -1.0;
            sa = cmul(t, cadd(sa, {sgn / (n + 1), 0.0}));
            sb = cmul(t, cadd(sb, {sgn / ((double)n * (n + 1)), 0.0}));
        }
        *c_a = sa;
        *c_b = sb;
        return;
    }
    const cplx u = {(w - x_a) / h, eta / h};
    const cplx L = {log(hypot(u.re, u.im) / hypot(q.re, q.im)), atan2(u.im, u.re) - atan2(q.im, q.re)};
    const cplx qL = cmul(q, L), uL = cmul(u, L);
    *c_a = {1.0 - qL.re, -qL.im};
    *c_b = {uL.re - 1.0, uL.im};
}

__global__ void hilbert_table_kernel(const double* __restrict__ omega, int n_omega, const double* __restrict__ w,
                                     int n_w, double eta, double* __restrict__ M) {
    const int64_t total = (int64_t)n_w * n_omega;
    for (int64_t o = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; o < total; o += (int64_t)gridDim.x * blockDim.x) {
        const int k = (int)(o / n_omega), j = (int)(o - (int64_t)k * n_omega);
        const double wk = w[k];
        cplx m = {0.0, 0.0}, ca, cb;
        if (j > 0) {                     // A_j is the right end of segment j-1
            segment_coeffs(omega[j - 1], omega[j], wk, eta, &ca, &cb);
            m = cadd(m, cb);
        }
        if (j + 1 < n_omega) {           // and the left end of segment j
            segment_coeffs(omega[j], omega[j + 1], wk, eta, &ca, &cb);
            m = cadd(m, ca);
        }
        M[2 * o] = m.re;
        M[2 * o + 1] = m.im;
    }
}

// ---- out[R, n_w] = epilogue(A M^T): FP64 DMMA GEMM ---------------------------------------------------------------
// The real product C[R, 2 n_w] = A[R, n_omega] B[n_omega, 2 n_w] with B[j, 2k + p] = (Re, Im)_p M[k, j]: every C
// fragment of mma.m8n8k4 holds two adjacent columns of one row, i.e. Re and Im of one G_r(z_k), so the epilogue is
// register-local.  CTA tile 64 rows x 64 real columns (32 frequencies) x 32 omega points, four warps of 32 x 32,
// cp.async double buffering.  A rows are read with an arbitrary leading dimension (one analyzer slot of A_out in
// place), 8 bytes at a time; M rows are 16-byte complex pairs.  Out-of-range rows, columns and omega points are
// zero-filled by the copies (src-size 0), so the products of the padding are exact zeros.
constexpr int HB_BM = 64, HB_BN = 32, HB_BK = 32, HB_THREADS = 128;
constexpr int HB_AS_LD = HB_BK + 4;          // A tile rows: fragment loads hit 16 banks x 2 wavefronts
constexpr int HB_BS_LD = 2 * HB_BK + 8;      // B tile: one complex column of M per row, (re, im) interleaved
constexpr int HB_STAGE = HB_BM * HB_AS_LD + HB_BN * HB_BS_LD;
constexpr int HB_SMEM = 2 * HB_STAGE * (int)sizeof(double);

__device__ __forceinline__ void cp_async8_zfill(void* smem_dst, const void* gmem_src, bool valid) {
    const uint32_t d = static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst));
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(d), "l"(gmem_src), "r"(valid ? 8 : 0));
}
__device__ __forceinline__ void cp_async16_zfill(void* smem_dst, const void* gmem_src, bool valid) {
    const uint32_t d = static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst));
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(d), "l"(gmem_src), "r"(valid ? 16 : 0));
}
__device__ __forceinline__ void cp_async_wait_one() { asm volatile("cp.async.wait_group 1;\n" ::: "memory"); }

__global__ void __launch_bounds__(HB_THREADS) hilbert_apply_kernel(
        const double* __restrict__ A, int64_t lda, int R, const double* __restrict__ M, int n_omega, int n_w,
        const double* __restrict__ w, double eta, int mode, const double* __restrict__ scale,
        const double* __restrict__ shift, double* __restrict__ out) {
    extern __shared__ __align__(16) double hb_smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int m0 = blockIdx.y * HB_BM, c0 = blockIdx.x * HB_BN;      // first row, first complex column (frequency)
    const int nk = (n_omega + HB_BK - 1) / HB_BK;

    auto load = [&](int stage, int kt) {
        double* As = hb_smem + stage * HB_STAGE;
        double* Bs = As + HB_BM * HB_AS_LD;
        const int k0 = kt * HB_BK;
#pragma unroll
        for (int i = 0; i < HB_BM * HB_BK / HB_THREADS; ++i) {
            const int e = tid + i * HB_THREADS, r = e / HB_BK, c = e % HB_BK;
            const bool ok = (m0 + r < R) && (k0 + c < n_omega);
            const double* src = ok ? A + (int64_t)(m0 + r) * lda + (k0 + c) : A;
            cp_async8_zfill(As + r * HB_AS_LD + c, src, ok);
        }
#pragma unroll
        for (int i = 0; i < HB_BN * HB_BK / HB_THREADS; ++i) {
            const int e = tid + i * HB_THREADS, cc = e / HB_BK, j = e % HB_BK;
            const bool ok = (c0 + cc < n_w) && (k0 + j < n_omega);
            const double* src = ok ? M + 2 * ((int64_t)(c0 + cc) * n_omega + (k0 + j)) : M;
            cp_async16_zfill(Bs + cc * HB_BS_LD + 2 * j, src, ok);
        }
        cp_async_commit();
    };

    const int wm = (warp & 1) * 32;              // warp's first row in the tile
    const int wc = (warp >> 1) * 16;             // warp's first complex column in the tile
    double acc[4][4][2];
#pragma unroll
    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;

    load(0, 0);
    for (int kt = 0; kt < nk; ++kt) {
        if (kt + 1 < nk) {
            load((kt + 1) & 1, kt + 1);
            cp_async_wait_one();
        } else {
            cp_async_wait_all();
        }
        __syncthreads();
        const double* As = hb_smem + (kt & 1) * HB_STAGE;
        const double* Bs = As + HB_BM * HB_AS_LD;
#pragma unroll
        for (int ks = 0; ks < HB_BK / 4; ++ks) {
            double a[4], b[4];
#pragma unroll
            for (int mi = 0; mi < 4; ++mi) a[mi] = As[(wm + mi * 8 + (lane >> 2)) * HB_AS_LD + ks * 4 + (lane & 3)];
            // B fragment element (k = lane % 4, n = lane / 4): complex column n / 2, part n % 2
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
                b[ni] = Bs[(wc + ni * 4 + (lane >> 3)) * HB_BS_LD + 2 * (ks * 4 + (lane & 3)) + ((lane >> 2) & 1)];
#pragma unroll
            for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                for (int ni = 0; ni < 4; ++ni) dmma(acc[mi][ni], a[mi], b[ni]);
        }
        __syncthreads();
    }

    // epilogue: C fragment (row lane / 4, columns 2 (lane % 4) + {0, 1}) = (Re, Im) G_r(z_k)
#pragma unroll
    for (int mi = 0; mi < 4; ++mi) {
        const int r = m0 + wm + mi * 8 + (lane >> 2);
        if (r >= R) continue;
        const double sc = (mode == 1 && scale) ? scale[r] : 1.0;
        const double sh = shift ? shift[r] : 0.0;
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) {
            const int k = c0 + wc + ni * 4 + (lane & 3);
            if (k >= n_w) continue;
            double gr = acc[mi][ni][0], gi = acc[mi][ni][1];
            if (mode == 1) {
                gr = fma(sc, gr, sh);
                gi = sc * gi;
            } else if (mode == 2) {                 // z + shift - 1/G
                const double d = gr * gr + gi * gi;
                const double ir = gr / d, ii = -gi / d;
                gr = w[k] + sh - ir;
                gi = eta - ii;
            }
            *reinterpret_cast<double2*>(out + 2 * ((int64_t)r * n_w + k)) = make_double2(gr, gi);
        }
    }
}

}  // namespace

}  // namespace mx

using namespace mx;

extern "C" {

int mx_hilbert_table(const double* omega, int32_t n_omega, const double* w, int32_t n_w, double eta, double* M,
                     void* stream) {
    if (!omega || !w || !M || n_omega < 2 || n_w < 1 || !(eta > 0.0)) return MX_ERR_BAD_ARG;
    const int64_t total = (int64_t)n_w * n_omega;
    const int grid = (int)((total + 255) / 256 < 4736 ? (total + 255) / 256 : 4736);
    hilbert_table_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(omega, n_omega, w, n_w, eta, M);
    return cudaGetLastError() == cudaSuccess ? MX_OK : MX_ERR_CUDA;
}

int mx_hilbert_apply(const double* A, int64_t lda, int32_t R, const double* M, int32_t n_omega, int32_t n_w,
                     const double* w, double eta, int32_t mode, const double* scale, const double* shift, double* out,
                     void* stream) {
    if (R == 0) return MX_OK;
    if (!A || !M || !out || R < 0 || n_omega < 1 || n_w < 1 || lda < n_omega || mode < 0 || mode > 2)
        return MX_ERR_BAD_ARG;
    if (mode == 2 && (!w || !(eta > 0.0))) return MX_ERR_BAD_ARG;
    if ((reinterpret_cast<uintptr_t>(M) & 15) != 0 || (reinterpret_cast<uintptr_t>(out) & 15) != 0 ||
        (reinterpret_cast<uintptr_t>(A) & 7) != 0)
        return MX_ERR_BAD_ARG;
    const int64_t row_tiles = ((int64_t)R + HB_BM - 1) / HB_BM, col_tiles = ((int64_t)n_w + HB_BN - 1) / HB_BN;
    if (row_tiles > 65535 || col_tiles > 2147483647) return MX_ERR_UNSUPPORTED;
    if (cudaFuncSetAttribute(hilbert_apply_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, HB_SMEM) != cudaSuccess)
        return MX_ERR_CUDA;
    hilbert_apply_kernel<<<dim3((unsigned)col_tiles, (unsigned)row_tiles), HB_THREADS, HB_SMEM, (cudaStream_t)stream>>>(
        A, lda, R, M, n_omega, n_w, w, eta, mode, scale, shift, out);
    return cudaGetLastError() == cudaSuccess ? MX_OK : MX_ERR_CUDA;
}

}  // extern "C"

// Batched shifted matrix inversion for the inversion method of matrix-valued self-energies:
//   mode 0: Y(b,k) = ((z_k + C_b) 1 - X(b,k))^{-1}      G_aux from Sigma on the Matsubara axis
//   mode 1: Y(b,k) = (z_k + C_b) 1 - X(b,k)^{-1}        Sigma from G_aux(w + i eta)
// for X[B, M, M, n_z] complex with the frequency innermost.  One thread per (b, k): for a fixed element (i, j) the lanes
// of a warp read consecutive k, i.e. consecutive 16-byte complex values, so every load and store is coalesced.  The
// inversion is FP64 Gauss-Jordan with partial pivoting by modulus in a fixed operation order, so Y(b,k) depends on
// X(b,k), z_k and C_b only, never on the rest of the batch.  The kernel moves 16 M^2 bytes per (b, k) each way and does
// O(M^3) flops on them: memory-bound for every M it takes.
#include "mx_common.cuh"

namespace mx {

namespace {

constexpr int RS_THREADS = 128;               // matrix in registers
constexpr int RS_SMEM_THREADS = 64;           // matrix in a shared-memory slab (M >= RS_SMEM_MIN), <= 128 registers
constexpr int RS_SMEM_MIN = 5;                // ptxas -v: in registers M = 5 lands on the stack and M = 6 spills
constexpr int RS_GRID_CAP = 148 * 32;

struct cplx {
    double re, im;
};

// 1 / b by Smith's method with the operation order of numpy's complex division 1.0 / b (no contracted FMAs): a
// diagonal matrix gives the bits of the scalar self-energy path, which forms G_aux = 1 / (i nu + C - Sigma) with numpy.
__device__ __forceinline__ cplx crecip(cplx b) {
    cplx r;
    if (fabs(b.re) >= fabs(b.im)) {
        const double rat = b.im / b.re, scl = 1.0 / __dadd_rn(b.re, __dmul_rn(b.im, rat));
        r.re = __dmul_rn(__dadd_rn(1.0, __dmul_rn(0.0, rat)), scl);
        r.im = __dmul_rn(__dsub_rn(0.0, rat), scl);
    } else {
        const double rat = b.re / b.im, scl = 1.0 / __dadd_rn(b.im, __dmul_rn(b.re, rat));
        r.re = __dmul_rn(__dadd_rn(rat, 0.0), scl);
        r.im = __dmul_rn(__dsub_rn(__dmul_rn(0.0, rat), 1.0), scl);
    }
    return r;
}

__device__ __forceinline__ cplx cmul(cplx a, cplx b) { return {a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re}; }
__device__ __forceinline__ double cabs2(cplx a) { return a.re * a.re + a.im * a.im; }

// The M x M matrix of one thread: registers (every index a compile-time constant after unrolling) or a shared-memory
// slab laid out [M * M][blockDim], so that the lanes of a warp touch consecutive 16-byte words and no bank twice.
template <int M>
struct RegMatrix {
    cplx a[M * M];
    __device__ __forceinline__ cplx& operator()(int i, int j) { return a[i * M + j]; }
};

template <int M>
struct SmemMatrix {
    cplx* base;
    int stride;
    __device__ __forceinline__ cplx& operator()(int i, int j) { return base[(i * M + j) * stride]; }
};

// In-place Gauss-Jordan inversion with partial pivoting by modulus (the first row of largest |a_rk|^2 wins).  Every loop
// is unrolled: a row or column swap is a predicated exchange with compile-time indices, so a register matrix stays in
// registers.  Returns false for an exactly zero pivot.
template <int M, class Mat>
__device__ __forceinline__ bool gauss_jordan(Mat& a) {
    uint32_t perm = 0;                        // pivot row of step k in bits 3k..3k+2 (M <= 8)
    bool ok = true;
#pragma unroll
    for (int k = 0; k < M; ++k) {
        int p = k;
        double best = cabs2(a(k, k));
#pragma unroll
        for (int r = k + 1; r < M; ++r) {
            const double v = cabs2(a(r, k));
            if (v > best) { best = v; p = r; }
        }
        perm |= (uint32_t)p << (3 * k);
#pragma unroll
        for (int r = k + 1; r < M; ++r) {
            if (p == r) {
#pragma unroll
                for (int j = 0; j < M; ++j) {
                    const cplx t = a(k, j);
                    a(k, j) = a(r, j);
                    a(r, j) = t;
                }
            }
        }
        const cplx piv = a(k, k);
        ok = ok && (piv.re != 0.0 || piv.im != 0.0);
        const cplx inv = crecip(piv);
        a(k, k) = inv;
#pragma unroll
        for (int j = 0; j < M; ++j)
            if (j != k) a(k, j) = cmul(a(k, j), inv);
#pragma unroll
        for (int r = 0; r < M; ++r) {
            if (r == k) continue;
            const cplx f = a(r, k);
            const cplx g = cmul(f, inv);
            a(r, k) = {-g.re, -g.im};
#pragma unroll
            for (int j = 0; j < M; ++j) {
                if (j == k) continue;
                const cplx d = cmul(f, a(k, j));
                a(r, j) = {a(r, j).re - d.re, a(r, j).im - d.im};
            }
        }
    }
    // the row exchanges of the elimination are column exchanges of the inverse, undone in reverse order
#pragma unroll
    for (int k = M - 2; k >= 0; --k) {
#pragma unroll
        for (int c = k + 1; c < M; ++c) {
            if (((perm >> (3 * k)) & 7u) == (uint32_t)c) {
#pragma unroll
                for (int i = 0; i < M; ++i) {
                    const cplx t = a(i, k);
                    a(i, k) = a(i, c);
                    a(i, c) = t;
                }
            }
        }
    }
    return ok;
}

template <int M, class Mat>
__device__ __forceinline__ void resolve_one(Mat& a, const double* X, int64_t e0, int64_t es, const double2* z, int k,
                                            double c, int mode, double* Y) {
    const double2 zk = z[k];
    const cplx s = {zk.x + c, zk.y};
    bool finite = true;
#pragma unroll
    for (int i = 0; i < M; ++i)
#pragma unroll
        for (int j = 0; j < M; ++j) {
            const double2 x = *reinterpret_cast<const double2*>(X + 2 * (e0 + (i * M + j) * es));
            finite = finite && isfinite(x.x) && isfinite(x.y);
            a(i, j) = (mode == 0) ? cplx{(i == j ? s.re : 0.0) - x.x, (i == j ? s.im : 0.0) - x.y} : cplx{x.x, x.y};
        }
    const bool ok = gauss_jordan<M>(a) && finite;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
#pragma unroll
    for (int i = 0; i < M; ++i)
#pragma unroll
        for (int j = 0; j < M; ++j) {
            cplx y = a(i, j);
            if (mode == 1) y = {(i == j ? s.re : 0.0) - y.re, (i == j ? s.im : 0.0) - y.im};
            if (!ok) y = {nan, nan};
            *reinterpret_cast<double2*>(Y + 2 * (e0 + (i * M + j) * es)) = make_double2(y.re, y.im);
        }
}

// X and Y may be the same buffer: each thread reads its whole matrix before it writes it, and no other thread touches it.
template <int M>
__global__ void __launch_bounds__(RS_THREADS) resolvent_reg_kernel(const double* X, int B, int n_z,
                                                                  const double2* __restrict__ z,
                                                                  const double* __restrict__ C, int mode, double* Y) {
    const int64_t total = (int64_t)B * n_z;
    for (int64_t o = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; o < total; o += (int64_t)gridDim.x * blockDim.x) {
        const int b = (int)(o / n_z), k = (int)(o - (int64_t)b * n_z);
        RegMatrix<M> a;
        resolve_one<M>(a, X, (int64_t)b * M * M * n_z + k, n_z, z, k, C ? C[b] : 0.0, mode, Y);
    }
}

template <int M>
__global__ void __launch_bounds__(RS_SMEM_THREADS, 8) resolvent_smem_kernel(const double* X, int B, int n_z,
                                                                        const double2* __restrict__ z,
                                                                        const double* __restrict__ C, int mode,
                                                                        double* Y) {
    extern __shared__ __align__(16) double rs_smem[];
    SmemMatrix<M> a{reinterpret_cast<cplx*>(rs_smem) + threadIdx.x, (int)blockDim.x};
    const int64_t total = (int64_t)B * n_z;
    for (int64_t o = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; o < total; o += (int64_t)gridDim.x * blockDim.x) {
        const int b = (int)(o / n_z), k = (int)(o - (int64_t)b * n_z);
        resolve_one<M>(a, X, (int64_t)b * M * M * n_z + k, n_z, z, k, C ? C[b] : 0.0, mode, Y);
    }
}

template <int M>
int launch_resolvent(const double* X, int B, int n_z, const double* z, const double* C, int mode, double* Y,
                     cudaStream_t stream) {
    const int64_t total = (int64_t)B * n_z;
    const double2* z2 = reinterpret_cast<const double2*>(z);
    if constexpr (M < RS_SMEM_MIN) {
        const int grid = (int)((total + RS_THREADS - 1) / RS_THREADS < RS_GRID_CAP ? (total + RS_THREADS - 1) / RS_THREADS
                                                                                  : RS_GRID_CAP);
        resolvent_reg_kernel<M><<<grid, RS_THREADS, 0, stream>>>(X, B, n_z, z2, C, mode, Y);
    } else {
        const int smem = M * M * (int)sizeof(cplx) * RS_SMEM_THREADS;
        if (cudaFuncSetAttribute(resolvent_smem_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) !=
            cudaSuccess)
            return MX_ERR_CUDA;
        const int64_t blocks = (total + RS_SMEM_THREADS - 1) / RS_SMEM_THREADS;
        const int grid = (int)(blocks < RS_GRID_CAP ? blocks : RS_GRID_CAP);
        resolvent_smem_kernel<M><<<grid, RS_SMEM_THREADS, smem, stream>>>(X, B, n_z, z2, C, mode, Y);
    }
    return cudaGetLastError() == cudaSuccess ? MX_OK : MX_ERR_CUDA;
}

}  // namespace

}  // namespace mx

using namespace mx;

extern "C" {

int mx_matrix_resolvent(const double* X, int32_t B, int32_t M, int32_t n_z, const double* z, const double* C,
                        int32_t mode, double* Y, void* stream) {
    if (M < 1 || M > MX_MAX_MATRIX) return MX_ERR_UNSUPPORTED;
    if (B < 0 || n_z < 0 || (mode != 0 && mode != 1)) return MX_ERR_BAD_ARG;
    if (B == 0 || n_z == 0) return MX_OK;
    if (!X || !z || !Y) return MX_ERR_BAD_ARG;
    if ((reinterpret_cast<uintptr_t>(X) & 15) != 0 || (reinterpret_cast<uintptr_t>(Y) & 15) != 0 ||
        (reinterpret_cast<uintptr_t>(z) & 15) != 0 || (reinterpret_cast<uintptr_t>(C) & 7) != 0)
        return MX_ERR_BAD_ARG;
    const cudaStream_t s = (cudaStream_t)stream;
    switch (M) {
        case 1: return launch_resolvent<1>(X, B, n_z, z, C, mode, Y, s);
        case 2: return launch_resolvent<2>(X, B, n_z, z, C, mode, Y, s);
        case 3: return launch_resolvent<3>(X, B, n_z, z, C, mode, Y, s);
        case 4: return launch_resolvent<4>(X, B, n_z, z, C, mode, Y, s);
        case 5: return launch_resolvent<5>(X, B, n_z, z, C, mode, Y, s);
        case 6: return launch_resolvent<6>(X, B, n_z, z, C, mode, Y, s);
        case 7: return launch_resolvent<7>(X, B, n_z, z, C, mode, Y, s);
        default: return launch_resolvent<8>(X, B, n_z, z, C, mode, Y, s);
    }
}

}  // extern "C"

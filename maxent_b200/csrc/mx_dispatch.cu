// Dispatch of the fused sweep over the compiled tile-count instantiations of the kernel.
#include "mx_common.cuh"
namespace mx2 {
int sweep2_nt4(const mx::SweepArgs&, cudaStream_t, bool, int*, int*);
int sweep2_nt5(const mx::SweepArgs&, cudaStream_t, bool, int*, int*);
int sweep2_nt6(const mx::SweepArgs&, cudaStream_t, bool, int*, int*);
int sweep2_nt7(const mx::SweepArgs&, cudaStream_t, bool, int*, int*);
int sweep2_nt8(const mx::SweepArgs&, cudaStream_t, bool, int*, int*);
int sweep2_nt9(const mx::SweepArgs&, cudaStream_t, bool, int*, int*);
int sweep2_nt10(const mx::SweepArgs&, cudaStream_t, bool, int*, int*);
int sweep2_nt12(const mx::SweepArgs&, cudaStream_t, bool, int*, int*);
int sweep2_nt16(const mx::SweepArgs&, cudaStream_t, bool, int*, int*);
int sweep2_nt20(const mx::SweepArgs&, cudaStream_t, bool, int*, int*);
int sweep2_nt24(const mx::SweepArgs&, cudaStream_t, bool, int*, int*);
int sweep2_nt28(const mx::SweepArgs&, cudaStream_t, bool, int*, int*);
int sweep2_nt32(const mx::SweepArgs&, cudaStream_t, bool, int*, int*);
long long sweep2_wide_doubles(int nt);
int sweep2_threads();
}  // namespace mx2

namespace mx {

int sweep_threads() { return mx2::sweep2_threads(); }

int64_t sweep_rows_doubles(int n_omega, int variant, int grid) {
    const int64_t rowlen = (int64_t)((n_omega + 7) / 8) * 8;
    return (int64_t)grid * (variant == MX_VARIANT_PLUSMINUS ? 2 : 1) * 9 * rowlen;
}
int64_t sweep_wide_stride(int n_sv) { return mx2::sweep2_wide_doubles(sweep_tiles(n_sv)); }
int64_t sweep_scratch_doubles(int n_sv, int n_omega, int variant, int grid) {
    return sweep_rows_doubles(n_omega, variant, grid) + (int64_t)grid * sweep_wide_stride(n_sv);
}

int dispatch_sweep(SweepArgs& a, cudaStream_t stream, bool query, int* o_smem, int* o_grid) {
    const int s = a.n_sv;
    if (s < 1) return MX_ERR_BAD_ARG;
    int pk = (s * (s + 1)) / 2;
    pk = (pk + 1) & ~1;
    a.pk = pk;
    if (s > MX_MAX_NSV) return MX_ERR_UNSUPPORTED;
    switch (sweep_tiles(s)) {
        case 4: return mx2::sweep2_nt4(a, stream, query, o_smem, o_grid);
        case 5: return mx2::sweep2_nt5(a, stream, query, o_smem, o_grid);
        case 6: return mx2::sweep2_nt6(a, stream, query, o_smem, o_grid);
        case 7: return mx2::sweep2_nt7(a, stream, query, o_smem, o_grid);
        case 8: return mx2::sweep2_nt8(a, stream, query, o_smem, o_grid);
        case 9: return mx2::sweep2_nt9(a, stream, query, o_smem, o_grid);
        case 10: return mx2::sweep2_nt10(a, stream, query, o_smem, o_grid);
        case 12: return mx2::sweep2_nt12(a, stream, query, o_smem, o_grid);
        case 16: return mx2::sweep2_nt16(a, stream, query, o_smem, o_grid);
        case 20: return mx2::sweep2_nt20(a, stream, query, o_smem, o_grid);
        case 24: return mx2::sweep2_nt24(a, stream, query, o_smem, o_grid);
        case 28: return mx2::sweep2_nt28(a, stream, query, o_smem, o_grid);
        default: return mx2::sweep2_nt32(a, stream, query, o_smem, o_grid);
    }
}
}  // namespace mx

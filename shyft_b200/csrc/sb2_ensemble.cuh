// sb2_ensemble.cuh -- the one kernel a forcing-ensemble run adds (sb2_run_ensemble, DESIGN.md section 3.7).
//
// The members of a forcing ensemble are stepped as one internal region of members x np cells: member e's copy of cell c is internal
// cell e * np + c, np = n rounded up to the 32-cell warp.  This kernel lays rows of the parent region's geometry ([rows][n], one
// buffer per member or one shared by all) out into that region's [rows][members * np]: each member's n columns, then np - n padding
// columns that repeat the member's last cell (inactive cells, which read their inputs but use none of them).  It places the
// interpolated forcing of every window, and the parent's state ([n_state][n], shared) at the start of a pass.
#pragma once
#include <cstdint>

namespace sb2 {

// dst[r][(e0 + e) * np + c] = src[e * src_member_stride + r * n + min(c, n - 1)] for e < gridDim.z, r < rows, c < np.  Consecutive
// threads take consecutive columns, so both sides are read and written in whole 32-column runs.
__global__ void ensemble_scatter_kernel(const double* __restrict__ src, int64_t src_member_stride, int64_t n, int64_t np, int64_t rows,
                                        double* __restrict__ dst, int64_t dst_cols, int64_t e0) {
    const int64_t c = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (c >= np) return;
    const int64_t e = blockIdx.z;
    const double* s = src + e * src_member_stride + (c < n ? c : n - 1);
    double* d = dst + (e0 + e) * np + c;
    for (int64_t r = blockIdx.y; r < rows; r += gridDim.y) d[r * dst_cols] = s[r * n];
}

}  // namespace sb2

// sb2_stats.cuh -- statistics readers over the resident [step][cell] series (SURVEY section 8f, item 1).
//
// Follows core/cell_model.h:194-406 (cell_statistics::sum_catchment_feature, average_catchment_feature and their *_value /
// catchment_feature forms) as api/api.h:178-1600 uses them (model.statistics.discharge(cids), .temperature(cids),
// gamma_snow_response.sca(cids), ...): a selection of cells (by catchment id or by cell index, empty = all) is summed, or
// averaged with the cell areas as weights (r += ts * area per cell, then r *= 1 / sum_area), step by step.
// The reference adds cell after cell; here a block reduces one step's row in a fixed tree (deterministic; differs from the
// sequential sum by rounding only: tests compare with the oracle at 1e-12, and with the exact sum within gamma(strides + 13) of the
// sum of |terms|, tests/test_gpu_statistics_paths.py).
#pragma once
#include <stdint.h>

#include "sb2_hbv.cuh"
#include "sb2_ptgsk.cuh"

namespace sb2 {

// out[t] = sum over selected cells of w[c] * f(v[t][c])   (w = nullptr: plain sum); one block per step row.
// f = identity, or (ae_scale != nullptr) the pot_ratio of actual_evapotranspiration_cell_response_statistics (api/api.h:1527-1541):
// 1 - exp(-m3s_to_mmh(kirchner_discharge, area) * 3 / ae_scale_factor) of the cell's instant Kirchner discharge.
__device__ __forceinline__ double stat_pot_ratio(double q_m3s, double area, double scale) {
    return 1.0 - sb_exp(-m3s_to_mmh(q_m3s, area) * 3.0 / scale);  // actual_evapotranspiration.h:40-43
}
__global__ void __launch_bounds__(256) stat_reduce_rows_kernel(const double* __restrict__ v /* [rows][n_cells] */, int64_t n_cells, int64_t rows,
                                                               const uint8_t* __restrict__ sel, const double* __restrict__ w,
                                                               const double* __restrict__ area, const double* __restrict__ ae_scale,
                                                               double* __restrict__ out /* [rows] */) {
    __shared__ double part[8];
    for (int64_t r = blockIdx.x; r < rows; r += gridDim.x) {
        const double* row = v + r * n_cells;
        double acc = 0.0;
        for (int64_t c = threadIdx.x; c < n_cells; c += blockDim.x)
            if (sel[c]) {
                const double x = ae_scale != nullptr ? stat_pot_ratio(row[c], area[c], ae_scale[c]) : row[c];
                acc += w != nullptr ? x * w[c] : x;
            }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, off);
        if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
            double s = 0.0;
            for (int k = 0; k < (blockDim.x >> 5); ++k) s += part[k];
            out[r] = s;
        }
        __syncthreads();
    }
}

// catchment_feature: the selected cells' values of one step, compacted in cell order (positions precomputed on the host)
__global__ void stat_gather_row_kernel(const double* __restrict__ row /* [n_cells] */, const int64_t* __restrict__ cells, int64_t n_sel,
                                       const double* __restrict__ area, const double* __restrict__ ae_scale, double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_sel) return;
    const int64_t c = cells[i];
    out[i] = ae_scale != nullptr ? stat_pot_ratio(row[c], area[c], ae_scale[c]) : row[c];
}
// ae.ae_scale_factor of every cell's parameter set (region parameter or catchment override)
__global__ void stat_cell_ae_scale_kernel(int64_t n_cells, const int32_t* __restrict__ pset, const PtgskParam* __restrict__ params,
                                          double* __restrict__ out) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c < n_cells) out[c] = params[pset[c]].ae_scale_factor;
}

__global__ void stat_cell_ae_scale_hbv_kernel(int64_t n_cells, const int32_t* __restrict__ pset, const HbvParam* __restrict__ params,
                                              double* __restrict__ out) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c < n_cells) out[c] = params[pset[c]].ae_scale_factor;
}
__global__ void stat_cell_ae_scale_ssk_kernel(int64_t n_cells, const int32_t* __restrict__ pset, const SskParam* __restrict__ params,
                                              double* __restrict__ out) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c < n_cells) out[c] = params[pset[c]].ae_scale_factor;
}
__global__ void stat_cell_ae_scale_hps_kernel(int64_t n_cells, const int32_t* __restrict__ pset, const HpsParam* __restrict__ params,
                                              double* __restrict__ out) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c < n_cells) out[c] = params[pset[c]].ae_scale_factor;
}

}  // namespace sb2

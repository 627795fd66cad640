// sb2_routing.cuh -- cell-to-river unit-hydrograph convolution and river-network accumulation as shared-memory kernels.
//
// Follows core/routing.h:326-383 (routing::model: cell_uhg, cell_output_m3s, local_inflow, upstream_inflow, output_m3s),
// core/routing.h:399-421 (make_uhg_from_gamma, host side in sb2_host.hpp) and the USE_ZERO convolution of
// core/time_series.h:966-975.  The reference recurses upstream per query; here rivers are levelled once on the host
// (leaves first) and every level is one launch, so each river is convolved exactly once.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <tuple>
#include <vector>

#include "sb2_host.hpp"

namespace sb2 {

constexpr int ROUTE_CELLS = 128;  // cells per chunk (= threads per block)
constexpr int ROUTE_TT = 64;      // time steps per block

// local_inflow[r][g0 + t] = sum over the river's cells (ascending cell order, 128 at a time) of sum_j w_c[j] * q_c[t-j], t in [0, n_rows).
// `q` points at row 0 of a [rows][n_cells] block that also has `hist` valid rows BEFORE row 0 (the tail of the previous
// window); rows further back are before the start of the axis or not needed and read as zero (USE_ZERO, time_series.h:966-975).
// uhg_w rows are w_stride apart; depth (>= every cell UHG length, <= w_stride) is the tile's history depth: the river UHGs that
// share the table may be longer, but they never go through this tile.
// blockIdx.z = member of a calibration batch: its q block, cell UHG ids and local inflow lie at z times q_stride, uhg_stride and
// local_stride (0, 0, 0 with one member).
// grid (time tiles, rivers, members); dynamic smem: (ROUTE_TT + depth - 1) * ROUTE_CELLS doubles
__global__ void __launch_bounds__(ROUTE_CELLS) route_local_inflow_kernel(const double* __restrict__ q, int64_t n_cells, int64_t n_rows, int64_t hist,
                                                                         int64_t g0, int64_t T, const int32_t* __restrict__ riv_ptr,
                                                                         const int32_t* __restrict__ riv_cells,
                                                                         const int32_t* __restrict__ cell_uhg_id /* per gathered cell */,
                                                                         const int32_t* __restrict__ uhg_len, const double* __restrict__ uhg_w,
                                                                         int w_stride, int depth, double* __restrict__ local /* [n_riv][T] */,
                                                                         int64_t q_stride, int64_t uhg_stride, int64_t local_stride) {
    extern __shared__ double sq[];  // [(ROUTE_TT + depth - 1)][ROUTE_CELLS]
    __shared__ double acc[ROUTE_TT];
    q += blockIdx.z * q_stride;
    cell_uhg_id += blockIdx.z * uhg_stride;
    local += blockIdx.z * local_stride;
    const int r = blockIdx.y;
    const int64_t t0 = (int64_t)blockIdx.x * ROUTE_TT;
    const int nt = int(min((int64_t)ROUTE_TT, n_rows - t0));
    const int rows = ROUTE_TT + depth - 1;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < ROUTE_TT) acc[threadIdx.x] = 0.0;
    for (int k0 = riv_ptr[r]; k0 < riv_ptr[r + 1]; k0 += ROUTE_CELLS) {
        const int nc = min(ROUTE_CELLS, riv_ptr[r + 1] - k0);
        __syncthreads();
        {
            const int c = threadIdx.x;
            const int64_t cell = c < nc ? riv_cells[k0 + c] : -1;
            for (int row = 0; row < rows; ++row) {
                const int64_t t = t0 - (depth - 1) + row;  // row of the block, may be negative (history)
                sq[row * ROUTE_CELLS + c] = (cell >= 0 && t >= -hist && t < n_rows && g0 + t >= 0) ? q[t * n_cells + cell] : 0.0;
            }
        }
        __syncthreads();
        // warp w reduces rows t = w, w+4, ...; lane l covers cells l, l+32, l+64, l+96
        for (int ti = warp; ti < nt; ti += ROUTE_CELLS / 32) {
            double s = 0.0;
            for (int c = lane; c < nc; c += 32) {
                const int id = cell_uhg_id[k0 + c];
                const int len = uhg_len[id];
                const double* w = uhg_w + (int64_t)id * w_stride;
                double v = 0.0;
                for (int j = 0; j < len; ++j) v += w[j] * sq[(ti + depth - 1 - j) * ROUTE_CELLS + c];
                s += v;
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off);
            if (lane == 0) acc[ti] += s;
        }
    }
    __syncthreads();
    if (threadIdx.x < nt) local[(int64_t)r * T + g0 + t0 + threadIdx.x] = acc[threadIdx.x];
}

// one network level: upstream[r][t] = sum of output[u][t] over upstream rivers u; output[r] = (local[r] + upstream[r]) (*) uhg_r
// blockIdx.z = member of a calibration batch: its local / upstream / output series lie at z times stride (0 with one member)
// grid (time tiles, rivers of this level, members); dynamic smem: (ROUTE_TT + max_len - 1) doubles
__global__ void __launch_bounds__(ROUTE_TT) route_river_level_kernel(const int32_t* __restrict__ level_rivers, const int32_t* __restrict__ up_ptr,
                                                                     const int32_t* __restrict__ up_idx, const int32_t* __restrict__ riv_uhg_id,
                                                                     const int32_t* __restrict__ uhg_len, const double* __restrict__ uhg_w, int max_len,
                                                                     int64_t T, const double* __restrict__ local, double* __restrict__ upstream,
                                                                     double* __restrict__ output, int64_t stride) {
    extern __shared__ double sin_[];  // input sum rows [t0 - (max_len-1), t0 + ROUTE_TT)
    local += blockIdx.z * stride;
    upstream += blockIdx.z * stride;
    output += blockIdx.z * stride;
    const int r = level_rivers[blockIdx.y];
    const int64_t t0 = (int64_t)blockIdx.x * ROUTE_TT;
    const int rows = ROUTE_TT + max_len - 1;
    for (int row = threadIdx.x; row < rows; row += blockDim.x) {
        const int64_t t = t0 - (max_len - 1) + row;
        double v = 0.0;
        if (t >= 0 && t < T) {
            double up = 0.0;
            for (int k = up_ptr[r]; k < up_ptr[r + 1]; ++k) up += output[(int64_t)up_idx[k] * T + t];
            if (row >= max_len - 1) upstream[(int64_t)r * T + t] = up;
            v = local[(int64_t)r * T + t] + up;
        }
        sin_[row] = v;
    }
    __syncthreads();
    const int64_t t = t0 + threadIdx.x;
    if (t < T) {
        const int id = riv_uhg_id[r];
        const int len = uhg_len[id];
        const double* w = uhg_w + (int64_t)id * max_len;
        double v = 0.0;
        for (int j = 0; j < len; ++j) v += w[j] * sin_[threadIdx.x + max_len - 1 - j];
        output[(int64_t)r * T + t] = v;
    }
}

// the last `rows` rows of each member's [rows_src][n_cells] block become the first rows of its block in the other buffer of a pair:
// dst[e][i] = src[e][i + shift] for i < rows * n_cells (the two never overlap, whatever rows and shift are).  grid (x, members)
__global__ void route_history_kernel(const double* __restrict__ src, double* __restrict__ dst, int64_t stride, int64_t shift, int64_t count) {
    src += blockIdx.y * stride + shift;
    dst += blockIdx.y * stride;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) dst[i] = src[i];
}

namespace routing_host {

struct DevBuf {
    void* p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    template <class T>
    T* upload(const std::vector<T>& h, cudaStream_t s) {
        if (h.empty()) return nullptr;
        if (cudaMalloc(&p, h.size() * sizeof(T)) != cudaSuccess) throw std::runtime_error("routing: device allocation failed");
        if (cudaMemcpyAsync(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, s) != cudaSuccess)
            throw std::runtime_error("routing: upload failed");
        return (T*)p;
    }
    template <class T>
    T* alloc(size_t n) {
        if (cudaMalloc(&p, std::max<size_t>(1, n) * sizeof(T)) != cudaSuccess) throw std::runtime_error("routing: device allocation failed");
        return (T*)p;
    }
};

struct UhgTable {
    std::map<std::tuple<int, double, double>, int> ids;
    std::vector<std::vector<double>> w;
    int id_of(int n_steps, double alpha, double beta) {
        auto key = std::make_tuple(n_steps, alpha, beta);
        auto f = ids.find(key);
        if (f != ids.end()) return f->second;
        w.push_back(host::make_uhg_from_gamma(n_steps, alpha, beta));
        return ids[key] = int(w.size()) - 1;
    }
};

}  // namespace routing_host

// Everything about a river network that does not depend on the simulated discharge: cells gathered per river, the
// unit-hydrograph table, upstream lists and levels.  cell_routing [members][n_cells][5] = routing id, distance, velocity, alpha,
// beta (velocity/alpha/beta from the cell's parameter set; one member for a model's own run, one per parameter set of a
// calibration batch, the routing id and distance the same in every member); rivers [n][6] = id, downstream id, distance,
// velocity, alpha, beta.  The members share one table (equal (steps, alpha, beta) are one entry, so a member's weights are the
// ones its own single-member plan has); d_cuhg is [members][n_gathered], max_len / cell_max_len the maxima over all members.
struct RoutingPlan {
    int n_riv = 0, max_len = 1, cell_max_len = 1, n_levels = 0, members = 1;
    int64_t n_gathered = 0;
    std::map<int64_t, int> ix_of_rid;
    std::vector<int> level_begin;
    routing_host::DevBuf b_ptr, b_cells, b_cuhg, b_len, b_w, b_ruhg, b_upp, b_upi, b_lvl;
    const int32_t *d_ptr = nullptr, *d_cells = nullptr, *d_cuhg = nullptr, *d_len = nullptr, *d_ruhg = nullptr, *d_upp = nullptr, *d_upi = nullptr,
                  *d_order = nullptr;
    const double* d_w = nullptr;
};

inline std::unique_ptr<RoutingPlan> build_routing_plan(const std::vector<double>& rivers, const std::vector<double>& cell_routing, int64_t n_cells,
                                                       int64_t dt_us, cudaStream_t stream) {
    using namespace routing_host;
    auto pl = std::make_unique<RoutingPlan>();
    const int n_riv = int(rivers.size() / 6);
    if (n_riv == 0) throw std::runtime_error("routing: the river network is empty");
    pl->n_riv = n_riv;
    const int members = int(cell_routing.size() / (5 * std::max<int64_t>(1, n_cells)));
    pl->members = std::max(1, members);
    for (int i = 0; i < n_riv; ++i) pl->ix_of_rid[int64_t(rivers[6 * i])] = i;
    UhgTable tab;
    std::vector<std::vector<int32_t>> cells_of(n_riv);
    std::vector<int32_t> cell_uhg(size_t(pl->members) * n_cells, 0);
    for (int e = 0; e < members; ++e) {
        const double* cr = cell_routing.data() + size_t(e) * n_cells * 5;
        for (int64_t c = 0; c < n_cells; ++c) {
            const int64_t id = int64_t(cr[5 * c]);
            if (id <= 0) continue;
            auto f = pl->ix_of_rid.find(id);
            if (f == pl->ix_of_rid.end()) throw std::runtime_error("river network: river id " + std::to_string(id) + " not found");
            if (e == 0) cells_of[f->second].push_back(int32_t(c));
            cell_uhg[size_t(e) * n_cells + c] = tab.id_of(host::uhg_steps(cr[5 * c + 1], cr[5 * c + 2], dt_us), cr[5 * c + 3], cr[5 * c + 4]);
        }
    }
    for (auto& w : tab.w) pl->cell_max_len = std::max(pl->cell_max_len, int(w.size()));
    std::vector<int32_t> riv_ptr(n_riv + 1, 0), riv_cells, riv_uhg(n_riv);
    for (int r = 0; r < n_riv; ++r) {
        for (auto c : cells_of[r]) riv_cells.push_back(c);
        riv_ptr[r + 1] = int32_t(riv_cells.size());
        riv_uhg[r] = tab.id_of(host::uhg_steps(rivers[6 * r + 2], rivers[6 * r + 3], dt_us), rivers[6 * r + 4], rivers[6 * r + 5]);
    }
    pl->n_gathered = int64_t(riv_cells.size());
    std::vector<int32_t> gathered_uhg(size_t(pl->members) * riv_cells.size());
    for (int e = 0; e < pl->members; ++e)
        for (size_t k = 0; k < riv_cells.size(); ++k) gathered_uhg[e * riv_cells.size() + k] = cell_uhg[size_t(e) * n_cells + riv_cells[k]];
    for (auto& w : tab.w) pl->max_len = std::max(pl->max_len, int(w.size()));
    // the shared-memory tiles: cell discharge of the local-inflow kernel, input sum of the river-level kernel
    if (size_t(ROUTE_TT + pl->cell_max_len - 1) * ROUTE_CELLS * sizeof(double) > 200 * 1024)
        throw std::runtime_error("routing: cell unit hydrograph too long for the shared-memory tile");
    if (size_t(ROUTE_TT + pl->max_len - 1) * sizeof(double) > 200 * 1024)
        throw std::runtime_error("routing: river unit hydrograph too long for the shared-memory tile");
    std::vector<int32_t> uhg_len(tab.w.size());
    std::vector<double> uhg_w(tab.w.size() * pl->max_len, 0.0);
    for (size_t i = 0; i < tab.w.size(); ++i) {
        uhg_len[i] = int32_t(tab.w[i].size());
        std::copy(tab.w[i].begin(), tab.w[i].end(), uhg_w.begin() + i * pl->max_len);
    }
    // upstream lists (ascending river id, routing.h:205-213) and levels (a river's level = 1 + max level of its upstreams)
    std::vector<std::vector<int32_t>> ups(n_riv);
    for (auto& kv : pl->ix_of_rid) {  // map order = ascending id
        const int64_t down = int64_t(rivers[6 * kv.second + 1]);
        if (down > 0) {
            auto f = pl->ix_of_rid.find(down);
            if (f == pl->ix_of_rid.end()) throw std::runtime_error("river network: downstream river id not found");
            ups[f->second].push_back(kv.second);
        }
    }
    std::vector<int> level(n_riv, -1);
    for (int pass = 0; pass <= n_riv; ++pass) {
        bool changed = false;
        for (int r = 0; r < n_riv; ++r) {
            if (level[r] >= 0) continue;
            int lv = 0;
            bool ready = true;
            for (auto u : ups[r]) { if (level[u] < 0) { ready = false; break; } lv = std::max(lv, level[u] + 1); }
            if (ready) { level[r] = lv; pl->n_levels = std::max(pl->n_levels, lv + 1); changed = true; }
        }
        if (!changed) break;
    }
    for (int r = 0; r < n_riv; ++r)
        if (level[r] < 0) throw std::runtime_error("river network: cycle detected");
    std::vector<int32_t> up_ptr(n_riv + 1, 0), up_idx, order;
    for (int r = 0; r < n_riv; ++r) { for (auto u : ups[r]) up_idx.push_back(u); up_ptr[r + 1] = int32_t(up_idx.size()); }
    pl->level_begin.assign(pl->n_levels + 1, 0);
    for (int lv = 0; lv < pl->n_levels; ++lv) {
        for (int r = 0; r < n_riv; ++r) if (level[r] == lv) order.push_back(r);
        pl->level_begin[lv + 1] = int(order.size());
    }
    pl->d_ptr = pl->b_ptr.upload(riv_ptr, stream);
    pl->d_cells = pl->b_cells.upload(riv_cells, stream);
    pl->d_cuhg = pl->b_cuhg.upload(gathered_uhg, stream);
    pl->d_len = pl->b_len.upload(uhg_len, stream);
    pl->d_w = pl->b_w.upload(uhg_w, stream);
    pl->d_ruhg = pl->b_ruhg.upload(riv_uhg, stream);
    pl->d_upp = pl->b_upp.upload(up_ptr, stream);
    pl->d_upi = pl->b_upi.upload(up_idx, stream);
    pl->d_order = pl->b_lvl.upload(order, stream);
    if (cudaStreamSynchronize(stream) != cudaSuccess) throw std::runtime_error("routing: upload failed");
    return pl;
}

// cell -> river: the local inflow of every river over block rows [0, n_rows) = global steps [g0, g0 + n_rows); with members > 1,
// member e's block row 0 is at d_q_row0 + e * q_stride and its local inflow [n_riv][T] at d_local + e * n_riv * T
inline void routing_local_inflow(const RoutingPlan& pl, const double* d_q_row0, int64_t n_cells, int64_t n_rows, int64_t hist, int64_t g0, int64_t T,
                                 double* d_local, cudaStream_t stream, int64_t* launches, int members = 1, int64_t q_stride = 0) {
    if (members > pl.members) throw std::runtime_error("routing: more members than the plan has unit hydrographs for");
    const size_t smem = size_t(ROUTE_TT + pl.cell_max_len - 1) * ROUTE_CELLS * sizeof(double);
    if (smem > 48 * 1024) cudaFuncSetAttribute(route_local_inflow_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    const unsigned tiles = unsigned((n_rows + ROUTE_TT - 1) / ROUTE_TT);
    route_local_inflow_kernel<<<dim3(tiles, pl.n_riv, members), ROUTE_CELLS, smem, stream>>>(
        d_q_row0, n_cells, n_rows, hist, g0, T, pl.d_ptr, pl.d_cells, pl.d_cuhg, pl.d_len, pl.d_w, pl.max_len, pl.cell_max_len, d_local,
        members > 1 ? q_stride : 0, members > 1 ? pl.n_gathered : 0, members > 1 ? int64_t(pl.n_riv) * T : 0);
    ++*launches;
    if (cudaGetLastError() != cudaSuccess) throw std::runtime_error("routing: kernel launch failed");
}

// river network, leaves first: upstream inflow and routed output of every river over the whole axis; d_local, d_up and d_out hold
// [members][n_riv][T]
inline void routing_network(const RoutingPlan& pl, int64_t T, const double* d_local, double* d_up, double* d_out, cudaStream_t stream, int64_t* launches,
                            int members = 1) {
    cudaMemsetAsync(d_up, 0, size_t(members) * pl.n_riv * T * sizeof(double), stream);
    const unsigned tiles = unsigned((T + ROUTE_TT - 1) / ROUTE_TT);
    const size_t smem = size_t(ROUTE_TT + pl.max_len - 1) * sizeof(double);
    if (smem > 48 * 1024) cudaFuncSetAttribute(route_river_level_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    for (int lv = 0; lv < pl.n_levels; ++lv) {
        const int cnt = pl.level_begin[lv + 1] - pl.level_begin[lv];
        route_river_level_kernel<<<dim3(tiles, cnt, members), ROUTE_TT, smem, stream>>>(pl.d_order + pl.level_begin[lv], pl.d_upp, pl.d_upi, pl.d_ruhg,
                                                                                       pl.d_len, pl.d_w, pl.max_len, T, d_local, d_up, d_out,
                                                                                       int64_t(pl.n_riv) * T);
        ++*launches;
    }
    if (cudaGetLastError() != cudaSuccess) throw std::runtime_error("routing: kernel launch failed");
}

}  // namespace sb2

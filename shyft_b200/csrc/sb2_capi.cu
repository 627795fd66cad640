// sb2_capi.cu -- the C ABI of include/shyft_b200.h over the sm_100a kernels.
//
// Mirrors the member surface of region_model<cell_t> (core/region_model.h:211-1049): construction and catchment
// indexing (:233-249,283-291), parameters (:646-708), filter (:715-729), states (:784-837), interpolate (:397-527),
// run_cells (:578-597), catchment_discharges/charges (:873-900).  Host code here only packs/unpacks structure-of-arrays
// data, builds the small station-side operators and launches kernels; there is no CPU compute path.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <memory>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/shyft_b200.h"
#include "sb2_host.hpp"
#include "sb2_interp.cuh"
#include "sb2_ptgsk.cuh"
#include "sb2_hbv.cuh"
#include "sb2_ptssk.cuh"
#include "sb2_pthpsk.cuh"
#include "sb2_routing.cuh"
#include <nvtx3/nvToolsExt.h>  // header-only; ranges are no-ops unless a profiler is attached
#include "sb2_unit.cuh"
#include "sb2_goal.cuh"
#include "sb2_stats.cuh"

using namespace sb2;

extern "C" int sb2_river_flows(sb2_model* m, int64_t rid, int64_t start_step, int64_t n_steps, double* local_inflow, double* upstream_inflow,
                               double* output);

namespace {

struct Error : std::runtime_error { using std::runtime_error::runtime_error; };

#define CUDA_OK(expr)                                                                                              \
    do {                                                                                                           \
        cudaError_t e_ = (expr);                                                                                   \
        if (e_ != cudaSuccess) throw Error(std::string("CUDA error: ") + cudaGetErrorString(e_) + " at " #expr);   \
    } while (0)

thread_local std::string g_create_error;

// Freed device buffers of >= 1 MB are parked (per device, by size, up to 40 % of the device memory) and handed back to the next allocation of the same
// size: re-initialising a model's environment drops and re-creates GB-sized windows, and cudaFree / cudaMalloc of those cost
// ~150 ms per run_interpolation + run_cells cycle (bench.py e2e leg).  A failed cudaMalloc empties the pool and retries.
struct DevicePool {
    std::mutex mu;
    std::map<std::pair<int, size_t>, std::vector<void*>> parked;
    size_t parked_bytes = 0, limit = 0;
    static DevicePool& get() { static DevicePool p; return p; }
    void* take(size_t bytes) {
        int dev = 0;
        cudaGetDevice(&dev);
        std::lock_guard<std::mutex> g(mu);
        auto f = parked.find({dev, bytes});
        if (f == parked.end() || f->second.empty()) return nullptr;
        void* p = f->second.back();
        f->second.pop_back();
        parked_bytes -= bytes;
        return p;
    }
    bool park(void* p, size_t bytes) {
        if (bytes < (1u << 20)) return false;
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceSynchronize();  // what cudaFree would do: nothing in flight may still touch the buffer when another stream takes it
        std::lock_guard<std::mutex> g(mu);
        if (limit == 0) {  // 40 % of the device's memory (72 GB on a B200: the window buffers and scratch of a 4 096-step window are 50 GB)
            size_t free_b = 0, total_b = 0;
            limit = (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && total_b > 0) ? total_b / 5 * 2 : (12ULL << 30);
        }
        if (parked_bytes + bytes > limit) return false;
        parked[{dev, bytes}].push_back(p);
        parked_bytes += bytes;
        return true;
    }
    void flush() {  // current device only
        int dev = 0;
        cudaGetDevice(&dev);
        std::lock_guard<std::mutex> g(mu);
        for (auto& kv : parked)
            if (kv.first.first == dev) {
                for (void* p : kv.second) { cudaFree(p); parked_bytes -= kv.first.second; }
                kv.second.clear();
            }
    }
};

// Red zones (diagnostic, SB2_GUARD=1 in the environment): compute-sanitizer is not available on every GPU pool, so the library can check
// itself for out-of-bounds WRITES -- every device buffer is then allocated with 4 KB of 0xA5 bytes in front of and behind it (the pool is
// bypassed), and sb2_check_guards() / every release verifies that the zones are intact.  tests/test_gpu_guards.py runs the multi-wave
// time-sliced step kernels, the TMA-staged interpolation, routing and the goal kernels this way.
struct GuardZones {
    static constexpr size_t Z = 4096;
    std::mutex mu;
    std::map<void*, size_t> live;  // user pointer -> user bytes
    int64_t violations = 0;
    std::string first;
    static GuardZones& get() { static GuardZones g; return g; }
    static bool on() { const char* e = std::getenv("SB2_GUARD"); return e && e[0] == '1'; }
    void* alloc(size_t bytes) {
        unsigned char* raw = nullptr;
        if (cudaMalloc((void**)&raw, bytes + 2 * Z) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        cudaMemset(raw, 0xA5, Z);
        cudaMemset(raw + Z + bytes, 0xA5, Z);
        std::lock_guard<std::mutex> g(mu);
        live[raw + Z] = bytes;
        return raw + Z;
    }
    bool owns(void* p) { std::lock_guard<std::mutex> g(mu); return live.count(p) != 0; }
    void check_one(void* p, size_t bytes) {  // mu held
        std::vector<unsigned char> h(2 * Z);
        cudaDeviceSynchronize();
        cudaMemcpy(h.data(), (unsigned char*)p - Z, Z, cudaMemcpyDeviceToHost);
        cudaMemcpy(h.data() + Z, (unsigned char*)p + bytes, Z, cudaMemcpyDeviceToHost);
        for (size_t i = 0; i < 2 * Z; ++i)
            if (h[i] != 0xA5) {
                ++violations;
                if (first.empty())
                    first = "red zone of a " + std::to_string(bytes) + "-byte device buffer overwritten " +
                            (i < Z ? std::to_string(Z - i) + " bytes before its start" : std::to_string(i - Z) + " bytes behind its end");
                break;
            }
    }
    void free(void* p) {
        std::lock_guard<std::mutex> g(mu);
        auto f = live.find(p);
        check_one(p, f->second);
        live.erase(f);
        cudaFree((unsigned char*)p - Z);
    }
    int64_t check_all() {
        std::lock_guard<std::mutex> g(mu);
        for (auto& kv : live) check_one(kv.first, kv.second);
        return violations;
    }
};

template <class T>
struct DevArray {  // library-owned device buffer
    T* p = nullptr;
    size_t n = 0;
    DevArray() {}
    DevArray(const DevArray&) = delete;
    DevArray& operator=(const DevArray&) = delete;
    ~DevArray() { release(); }
    void release() {
        if (p && GuardZones::get().owns(p)) GuardZones::get().free(p);
        else if (p && !DevicePool::get().park(p, n * sizeof(T))) cudaFree(p);
        p = nullptr; n = 0;
    }
    void resize(size_t count) {
        if (count == n) return;
        release();
        if (count && GuardZones::on()) {
            p = static_cast<T*>(GuardZones::get().alloc(count * sizeof(T)));
            if (!p) throw Error("device allocation of " + std::to_string(count * sizeof(T)) + " bytes (+ red zones) failed");
        } else if (count) {
            p = static_cast<T*>(DevicePool::get().take(count * sizeof(T)));
            if (!p) {
                cudaError_t e = cudaMalloc((void**)&p, count * sizeof(T));
                if (e != cudaSuccess) {  // give the parked buffers back to the driver and try once more
                    cudaGetLastError();
                    DevicePool::get().flush();
                    e = cudaMalloc((void**)&p, count * sizeof(T));
                }
                if (e != cudaSuccess) {
                    cudaGetLastError();
                    p = nullptr;
                    throw Error("device allocation of " + std::to_string(count * sizeof(T)) + " bytes failed: " + cudaGetErrorString(e));
                }
            }
        }
        n = count;
    }
    void ensure(size_t count) { if (count > n) resize(count); }
    void upload(const T* h, size_t count, cudaStream_t s) {
        resize(count);
        if (count) CUDA_OK(cudaMemcpyAsync(p, h, count * sizeof(T), cudaMemcpyHostToDevice, s));
    }
    void upload(const std::vector<T>& h, cudaStream_t s) { upload(h.data(), h.size(), s); }
};

// NVTX ranges around the phases of the ABI calls (nsys / ncu --nvtx timelines): interpolate, window i, forcing_terms / snow / response,
// catchment_reduce, routing
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    explicit NvtxRange(const std::string& name) { nvtxRangePushA(name.c_str()); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};

struct Source {  // one region_environment variable: geo-located series on the model axis (api/api.h:137-168)
    int64_t n_src = 0;
    std::vector<double> xyz;       // [src][3]
    std::vector<double> h_values;  // [T][src], host copy (BTK validity bookkeeping, single-source copy)
    DevArray<double> d_xyz, d_values;
    bool has_nonfinite = false;
};

struct IdwPlan {  // neighbour lists of one variable (inverse_distance.h:160-203), [k][cell] on the device
    bool valid = false;
    IdwParam p{};
    int64_t n_src = 0;
    DevArray<int32_t> idx, cnt;
    DevArray<double> w, f;
    bool dense_valid = false;      // dense operator for the all-finite case (tensor-core path)
    DevArray<double> dense, addc;  // [n_src][cells], [cells]
    DevArray<int32_t> ulist;       // station compaction of the dense apply kernel: [tiles][k_slots] union lists ...
    DevArray<uint8_t> ukc;         // ... and k-steps in use per tile (idw_union_plan_kernel)
    int kc_max = 0;                // the widest union, in k-steps
};

struct BtkOps {  // operators of one valid-station subset
    std::vector<int> valid;
    DevArray<double> omega, bm, E_beta_w, sz;
    DevArray<int32_t> valid_idx;
};

// Per-stack constants, indexed by SB2_PT_GS_K ... SB2_PT_HPS_K.  A model's parameter and state sizes are the sizes of the default vectors.
struct StackInfo {
    std::vector<double> parameter;  // parameter::get order, default-constructed values
    std::vector<double> state;      // flat ABI order, default-constructed cell state
    int n_state_series;             // state series the step kernel collects (ids of include/shyft_b200.h)
    int routing_velocity;           // parameter index of the routing velocity; alpha and beta follow
};
const StackInfo kStacks[5] = {
    // pt_gs_k::parameter() defaults, vector order; gamma_snow::state (gamma_snow.h:101-116) + kirchner.q (kirchner.h:124-126)
    {{-2.439, 0.966, -0.10, 1.5, -0.5, 2.0, 0.1, 1.0, 5.0, 5.0, 30.0, 0.9, 0.6, 5.0, 0.4, 0.4, 1.0, 0.0, 0.0, 0.2, 1.26,
      0.04,   100.0, 0.0,  6.0, 1.0,  7.0, 0.0, 221.0, 0.0, 1.0},
     {0.4, 0.1, 30000.0, 1.26, 0.0, 0.0, 0.0, 0.0, 0.1},
     9, 25},
    // pt_hs_k::parameter::get order (core/pt_hs_k.h:108-131); swe, sca, sp[5], sw[5] = 0 (hbv_snow.h:97-121) + kirchner.q
    {{-2.439, 0.966, -0.10, 1.5, 0.1, 0.0, 1.0, 0.0, 0.5, 6.0, 1.0, 0.2, 1.26, 1.0, 7.0, 0.0, 0.0, 1.0},
     {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.1},
     3 + 2 * HBV_NB, 13},
    // hbv_stack::parameter::get order (core/hbv_stack.h:127-155); swe, sca, sp[5], sw[5] = 0, soil.sm = 0 (hbv_soil.h:28), tank uz / lz (hbv_tank.h:32)
    {{300.0, 2.0, 150.0, 25.0, 0.5, 0.3, 0.8, 0.02, 0.1, 0.0, 1.0, 0.0, 0.5, 1.0, 0.2, 1.26, 6.0, 1.0, 7.0, 0.0, 0.0, 1.0},
     {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 20.0, 10.0},
     5 + 2 * HBV_NB, 17},
    // pt_ss_k::parameter::get order (core/pt_ss_k.h:90-117); skaugen::parameter defaults (core/skaugen.h:92-99);
    // skaugen::state (skaugen.h:121-124) + kirchner.q; num_units has no state series
    {{-2.439, 0.966, -0.10, 1.5, 40.77, 113.0, 0.1, 0.1, 0.16, 2.5, 0.14, 0.01, 1.0, 0.2, 1.26, 6.0, 1.0, 7.0, 0.0, 0.0, 1.0},
     {4.077, 40.77, 0.0, 0.0, 0.0, 0.0, 0.0, 0.1},
     7, 16},
    // pt_hps_k::parameter::get order (core/pt_hps_k.h:93-120); hbv_physical_snow::parameter defaults (:40-92);
    // hbv_physical_snow::state after distribute() (core/hbv_physical_snow.h:132-189): sp[5] = sw[5] = 0, albedo[5] = 0.4,
    // iso_pot_energy[5] = 0, surface_heat, swe, sca; + kirchner.q
    {{-2.439, 0.966, -0.10, 1.5, 0.1, 0.0, 0.5, 2.0, 1.0, 30.0, 0.9, 0.6, 5.0, 5.0, 5.0, 0.0, 6.0, 1.0, 0.2, 1.26, 1.0, 7.0, 0.0, 1.0},
     {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.4, 0.4, 0.4, 0.4, 0.4, 0.0, 0.0, 0.0, 0.0, 0.0, 30000.0, 0.0, 0.0, 0.1},
     4 + 4 * HBV_NB, 20},
};

inline int grid_for(int64_t n, int block) { return int((n + block - 1) / block); }

}  // namespace

#define SB2_HBV_UNIT_STEPS 64      // steps per time slice of the pt_ss_k / pt_hps_k / pt_hs_k / hbv_stack step kernels (128: within +-0.7 %)
#define SB2_DENSE_TILE_COMPACT 32  // steps staged per buffer, compacted inverse distance over 64-station rows

struct sb2_model {
    int stack = 0, device = 0;
    cudaStream_t stream = 0;
    std::string err;
    int64_t n = 0;
    std::vector<sb2_geo_cell> geo;
    std::vector<int64_t> cix_of_cell, cix_to_cid;
    std::map<int64_t, int64_t> cid_to_cix;
    int n_param = 0, n_state = 0;
    // parameters: region + per-catchment overrides (region_model.h:646-708)
    std::vector<double> region_param;
    std::map<int64_t, std::vector<double>> catch_param;
    bool param_dirty = true;
    std::vector<uint8_t> catchment_filter;  // by cix; empty = no filter
    bool filter_dirty = true;
    // static per-cell SoA
    DevArray<double> d_x, d_y, d_z, d_area, d_glacier, d_lake, d_reservoir, d_forest, d_slope;
    DevArray<int32_t> d_pset;
    DevArray<uint8_t> d_active;
    DevArray<PtgskParam> d_ptgsk_params;
    DevArray<HbvParam> d_hbv_params;
    DevArray<SskParam> d_ssk_params;
    DevArray<HpsParam> d_hps_params;
    // state [n_state][n] + the initial-state snapshot (region_model.h:313,593-594)
    DevArray<double> d_state, d_initial_state;
    bool has_initial = false;
    // time axis
    int64_t t0 = 0, dt = 0, T = 0;
    DevArray<int2> d_doy_soy;  // [T] (calendar day of year, seconds since the start of the year) of each period start, UTC
    std::vector<double> h_prior_gradient;
    DevArray<double> d_prior_gradient;
    // forcing [rows][n] per variable; rows cover steps [forcing_first, forcing_first + forcing_rows)
    DevArray<double> d_forcing[SB2_N_FORCING];
    int64_t forcing_first = 0, forcing_rows = 0;
    Source src[SB2_N_FORCING];
    // interpolation plan cache
    sb2_interpolation_parameter ip{};
    bool ip_valid = false;
    IdwPlan idw[SB2_N_FORCING];
    std::vector<std::unique_ptr<BtkOps>> btk_cache;
    DevArray<double> d_btk_kbuf, d_btk_beta, d_btk_resid;
    // collected series
    bool force_sparse_idw = false;  // diagnostics: run IDW through the per-neighbour kernel even when the dense operator applies
    int collect_bits = SB2_COLLECT_DISCHARGE;
    DevArray<double> d_resp[SB2_N_RESPONSE], d_st[SB2_N_STATE_SERIES];
    int64_t out_first = 0, out_rows = 0;  // response rows cover [out_first, out_first + out_rows); state series one more
    int64_t ran_first = 0, ran_steps = 0;
    DevArray<double> d_cq, d_cc;  // catchment sums [T][n_catch]
    // segmented catchment reduction
    DevArray<int32_t> d_slot, d_cat_ptr, d_cat_slots;
    int64_t n_slots = 0;
    DevArray<double> d_partial;
    DevArray<double> d_scr[5];  // pt_gs_k phase pipeline scratch [partial_steps][n] (sb2_ptgsk.cuh)
    DevArray<int> d_tickets;    // step kernel time split: [0] ticket counter, [1..] finished slices per cell group
    int partial_steps = 0;
    DevArray<int> d_error_flag, d_scan_flag;
    // routing (core/routing.h)
    std::vector<double> rivers;  // [n][6] id downstream distance velocity alpha beta
    std::unique_ptr<RoutingPlan> route;      // built on first use, dropped when the network or the parameters change
    DevArray<double> d_rlocal, d_rup, d_rout;  // [n_riv][T] local inflow / upstream inflow / routed output
    bool rlocal_valid = false, rnet_valid = false;
    DevArray<double> d_qhist;                // windowed runs: avg_discharge window preceded by the previous window's tail rows
    int64_t qhist_rows = 0;
    // calibration targets (core/model_calibration.h:242-329)
    struct Target {
        std::vector<double> obs;
        int64_t t0 = 0, dt = 0;
        std::vector<int64_t> cids;
        int64_t river_id = 0;
        double scale_factor = 1.0;
        int calc_mode = 0, property = 0;
        double s_r = 1.0, s_a = 1.0, s_b = 1.0;
        DevArray<double> d_obs, d_series;
        DevArray<int32_t> d_cix;
        bool aligned = true;                      // target periods are whole runs of model steps inside the model axis
        std::vector<int64_t> points;              // point axis: n + 1 period boundaries (empty: fixed_dt)
        DevArray<int64_t> d_points;
        DevArray<double> d_projected, d_scale;   // not aligned: the property (and its max-abs scale) projected onto the target axis
    };
    std::vector<std::unique_ptr<Target>> targets;
    DevArray<int32_t> d_cell_ptr, d_cell_of_catch;  // cells grouped by catchment (area-weighted snow means)
    DevArray<int64_t> d_axis_t;                     // the model axis' point times (projection of a property onto a foreign target axis)
    DevArray<int32_t> d_one_zero;
    // bookkeeping
    int64_t launches = 0;
    float last_step_ms = 0.f, last_interp_ms = 0.f;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};

    int64_t n_catch() const { return int64_t(cix_to_cid.size()); }
    void use_device() const { CUDA_OK(cudaSetDevice(device)); }
};

namespace {

template <class F>
int guarded(sb2_model* m, F&& f) {
    try {
        if (!m) throw Error("null model");
        m->use_device();
        f();
        return 0;
    } catch (const std::exception& e) {
        if (m) m->err = e.what();
        return 1;
    }
}
template <class F>
int guarded_c(const sb2_model* m, F&& f) { return guarded(const_cast<sb2_model*>(m), f); }

// ---- parameter tables ------------------------------------------------------------------------------------------
// vector order of pt_gs_k::parameter::set (core/pt_gs_k.h:77-112)
PtgskParam make_ptgsk_param(const double* v, int64_t dt_us) {
    PtgskParam p{};
    p.c1 = v[0]; p.c2 = v[1]; p.c3 = v[2];
    p.ae_scale_factor = v[3];
    p.tx = v[4]; p.wind_scale = v[5]; p.max_water = v[6]; p.wind_const = v[7];
    p.fast_albedo_decay_rate = v[8]; p.slow_albedo_decay_rate = v[9]; p.surface_magnitude = v[10];
    p.max_albedo = v[11]; p.min_albedo = v[12]; p.snowfall_reset_depth = v[13]; p.snow_cv = v[14]; p.glacier_albedo = v[15];
    p.p_corr_scale_factor = v[16];
    p.snow_cv_forest_factor = v[17]; p.snow_cv_altitude_factor = v[18];
    p.pt_albedo = v[19]; p.pt_alpha = v[20];
    p.initial_bare_ground_fraction = v[21];
    p.winter_end_day_of_year = int32_t(size_t(v[22]));
    p.calculate_iso_pot_energy = v[23] != 0.0 ? 1 : 0;
    p.gm_dtf = v[24];
    // v[25..27] routing velocity/alpha/beta: used by the routing kernels, not by the cell step
    p.n_winter_days = int32_t(size_t(v[28]));
    p.gm_direct_response = v[29];
    p.reservoir_direct_response_fraction = v[30];
    // gamma_snow.h:341-343, evaluated once per run instead of per step (same expressions, same libm)
    const double dt_in_days = (double(dt_us) / 1e6) / 86400.0;
    const double albedo_range = p.max_albedo - p.min_albedo;
    p.slow_albedo_decay_step = 0.5 * albedo_range * dt_in_days / p.slow_albedo_decay_rate;
    p.fast_albedo_decay_step = sb_pow(2.0, -dt_in_days / p.fast_albedo_decay_rate);
    // parameter-only divisors of the step with their reciprocals (div_by, sb2_math.cuh): the divisor expressions are the step's own
    p.inv_snowfall_reset_depth = make_inv_divisor(p.snowfall_reset_depth);
    p.inv_one_minus_y0 = make_inv_divisor(1.0 - p.initial_bare_ground_fraction);
    p.inv_max_water = make_inv_divisor(p.max_water);
    p.inv_ae_scale = make_inv_divisor(p.ae_scale_factor);
    return p;
}
// the step length the parameter tables derive their per-run constants from: 1 h until a time axis is set
int64_t param_dt(const sb2_model* m) { return m->dt > 0 ? m->dt : 3600000000LL; }

// the stack's parameter table of the vectors `sets` (parameter::get order): the region set and the catchment overrides of
// sync_parameters, or the members of a calibration batch, so a member's derived constants are the single evaluation's
template <class P>
void upload_params(sb2_model* m, const std::vector<const double*>& sets, DevArray<P>& d) {
    std::vector<P> tab;
    for (const double* v : sets) {
        if constexpr (std::is_same_v<P, PtgskParam>) tab.push_back(make_ptgsk_param(v, param_dt(m)));
        else if constexpr (std::is_same_v<P, SskParam>) tab.push_back(make_ssk_param(v));
        else if constexpr (std::is_same_v<P, HpsParam>) tab.push_back(make_hps_param(v, param_dt(m)));
        else tab.push_back(make_hbv_param(m->stack == SB2_HBV_STACK, v));
    }
    d.upload(tab, m->stream);
}

void sync_parameters(sb2_model* m) {
    if (!m->param_dirty) return;
    // set 0 = region parameter; one more set per catchment override (region_model.h:668-678)
    std::vector<int32_t> pset(m->n, 0);
    std::vector<const double*> sets{m->region_param.data()};
    std::map<int64_t, int32_t> set_of_cid;
    for (auto& kv : m->catch_param) { set_of_cid[kv.first] = int32_t(sets.size()); sets.push_back(kv.second.data()); }
    for (int64_t i = 0; i < m->n; ++i) {
        auto f = set_of_cid.find(m->geo[i].catchment_id);
        if (f != set_of_cid.end()) pset[i] = f->second;
    }
    m->d_pset.upload(pset, m->stream);
    if (m->stack == SB2_PT_GS_K) upload_params(m, sets, m->d_ptgsk_params);
    else if (m->stack == SB2_PT_SS_K) upload_params(m, sets, m->d_ssk_params);
    else if (m->stack == SB2_PT_HPS_K) upload_params(m, sets, m->d_hps_params);
    else upload_params(m, sets, m->d_hbv_params);
    CUDA_OK(cudaStreamSynchronize(m->stream));
    m->param_dirty = false;
}
void sync_filter(sb2_model* m) {
    if (!m->filter_dirty) return;
    if (m->catchment_filter.empty()) m->d_active.release();
    else {
        std::vector<uint8_t> a(m->n);
        for (int64_t i = 0; i < m->n; ++i) a[i] = m->catchment_filter[m->cix_of_cell[i]];
        m->d_active.upload(a, m->stream);
        CUDA_OK(cudaStreamSynchronize(m->stream));
    }
    m->filter_dirty = false;
}

// ---- catchment reduction layout: one slot per (warp, run of equal catchment_ix) -----------------------------
void build_slots(sb2_model* m) {
    std::vector<int32_t> slot(m->n);
    std::vector<std::vector<int32_t>> by_cat(m->n_catch());
    int32_t ns = 0;
    for (int64_t i = 0; i < m->n; ++i) {
        const bool head = (i % 32 == 0) || m->cix_of_cell[i] != m->cix_of_cell[i - 1];
        if (head) { by_cat[m->cix_of_cell[i]].push_back(ns); ++ns; }
        slot[i] = ns - 1;
    }
    m->n_slots = ns;
    std::vector<int32_t> ptr(m->n_catch() + 1, 0), flat;
    for (int64_t k = 0; k < m->n_catch(); ++k) {
        for (auto s : by_cat[k]) flat.push_back(s);
        ptr[k + 1] = int32_t(flat.size());
    }
    m->d_slot.upload(slot, m->stream);
    m->d_cat_ptr.upload(ptr, m->stream);
    m->d_cat_slots.upload(flat, m->stream);
}

void free_series(sb2_model* m) {
    for (auto& b : m->d_resp) b.release();
    for (auto& b : m->d_st) b.release();
    m->out_rows = 0;
}

// rows needed for the per-cell series of this stack / collect mode
bool wants_response(const sb2_model* m, int r) {
    const int bits = m->collect_bits;
    if (r <= SB2_R_CHARGE_M3S) return bits & 1;
    if (r <= SB2_R_SNOW_SWE) return bits & 2;
    if (r <= SB2_R_PE_OUTPUT) return bits & 4;
    return (bits & 4) && m->stack == SB2_HBV_STACK;  // soil_outflow
}

void ensure_series(sb2_model* m, int64_t first, int64_t rows) {
    if (m->out_rows != rows) free_series(m);  // a window buffer of the same size is reused as is
    for (int r = 0; r < SB2_N_RESPONSE; ++r) {
        if (wants_response(m, r)) m->d_resp[r].ensure(size_t(rows) * m->n);
        else m->d_resp[r].release();
    }
    for (int s = 0; s < SB2_N_STATE_SERIES; ++s) {
        if ((m->collect_bits & SB2_COLLECT_STATE) && s < kStacks[m->stack].n_state_series) m->d_st[s].ensure(size_t(rows + 1) * m->n);
        else m->d_st[s].release();
    }
    m->out_first = first;
    m->out_rows = rows;
}

void fill_nan(sb2_model* m, double* p, int64_t count) {
    if (!count) return;
    fill_kernel<<<std::min<int64_t>(grid_for(count, 256), 148 * 16), 256, 0, m->stream>>>(p, count, nan(""));
    ++m->launches;
}

// Time split of the snow / response kernels (sb2_ptgsk.cuh): worth it while a launch of whole-window blocks is only a few waves of
// the ~2 000 one-warp blocks a B200 holds of these kernels (100 000 cells = 3 125 blocks = 1.2-1.8 waves); with many waves the tail
// is small and the split only costs (ensembles: 6.8 -> 4.9 G cell-steps/s when split).
bool use_time_split(int64_t blocks_per_launch) { return blocks_per_launch < 16000; }

// cell groups (one-warp blocks) of the time-split step kernels; a tickets buffer holds [members] ticket counters, then
// [members][groups] finished slices
int step_groups(const sb2_model* m) {
    return m->stack == SB2_PT_GS_K ? std::max(grid_for(m->n, SB2_BLOCK_B), grid_for(m->n, SB2_BLOCK_C)) : grid_for(m->n, SB2_BLOCK);
}

// Where a chunk of the cell step reads and writes.  run_cells steps the model's own buffers as one member; a calibration batch
// steps `members` parameter sets at once, member e as grid layer e with its state, partial sums, catchment sums and scratch
// at e times the strides.
struct StepTarget {
    int members = 1;
    const PtgskParam* ptgsk_members = nullptr;  // the members' parameter sets, in place of the region set (null: no batch)
    const HbvParam* hbv_members = nullptr;
    const HpsParam* hps_members = nullptr;
    double* state = nullptr;
    double* partial = nullptr;
    double *cq = nullptr, *cc = nullptr;  // catchment sums [T][n_catch]
    DevArray<double>* scr = nullptr;      // pt_gs_k phase pipeline scratch, five arrays
    int64_t state_stride = 0, partial_stride = 0, catch_stride = 0, scr_stride = 0;
    int* tickets = nullptr;               // [members] + [members][step_groups]
    bool series = false;                  // write the model's collected series (m->collect_bits)
    // a batch with a routed target: avg_discharge / charge of the chunk's step i and cell c at q / charge + e * resp_stride + i * n
    double *q = nullptr, *charge = nullptr;
    int64_t resp_stride = 0;
};

// One chunk of steps [s0, s0 + chunk) for the model's stack: its step kernels, then catchment_reduce_kernel
void launch_step_chunk(sb2_model* m, const StepTarget& t, int64_t s0, int chunk, bool collect_end_state) {
    const int64_t n = m->n;
    const unsigned ne = unsigned(t.members);
    const bool gsk = m->stack == SB2_PT_GS_K;
    const int collect = t.series ? m->collect_bits : (t.q ? SB2_COLLECT_DISCHARGE : 0);
    // UPAR kernels: no catchment override and no member table -> every cell reads the region parameter set from the constant bank
    const bool upar = m->catch_param.empty() && !t.ptgsk_members && !t.hbv_members && !t.hps_members;
    // snow / response or run kernel in time slices handed out by ticket (see the kernels); the tickets are read only when split
    const int groups = step_groups(m);
    const bool split = use_time_split(int64_t(groups) * t.members);
    const int unit_steps = split ? (gsk ? SB2_UNIT_STEPS : SB2_HBV_UNIT_STEPS) : 0;
    const int n_slices = split ? grid_for(chunk, unit_steps) : 1;
    auto zero_tickets = [&] {
        if (split) CUDA_OK(cudaMemsetAsync(t.tickets, 0, size_t(t.members) * (1 + groups) * sizeof(int), m->stream));
    };
    // the fields all four *RunArgs share
    auto common = [&](auto& a) {
        const double dt_seconds = double(m->dt) / 1e6;
        a.n_cells = n;
        a.area = m->d_area.p; a.glacier = m->d_glacier.p; a.lake = m->d_lake.p; a.reservoir = m->d_reservoir.p;
        a.pset = m->d_pset.p; a.active = m->d_active.p; a.state = t.state;
        for (int v = 0; v < 5; ++v) a.f[v] = m->d_forcing[v].p + (s0 - m->forcing_first) * n;
        a.n_steps = chunk; a.first_step = s0;
        a.dt_seconds = dt_seconds; a.dt_hours = dt_seconds / 3600.0; a.dt_us = double(m->dt);
        fill_dopri_products(a.dt_hours, a.dtb);
        if (t.series) {
            for (size_t r = 0; r < std::size(a.resp); ++r) a.resp[r] = m->d_resp[r].p;
            for (size_t s = 0; s < std::size(a.st); ++s) a.st[s] = m->d_st[s].p;
            a.out_first_step = m->out_first;
        } else if (t.q) {
            a.resp[0] = t.q; a.resp[1] = t.charge;
            a.out_first_step = s0;
        }
        a.collect_end_state = collect_end_state ? 1 : 0;
        a.slot = m->d_slot.p; a.partial = t.partial; a.n_slots = m->n_slots; a.error_flag = m->d_error_flag.p;
        a.unit_steps = unit_steps; a.tickets = t.tickets; a.progress = t.tickets + t.members;
    };
    if (gsk) {
        PtgskRunArgs a{};
        common(a);
        a.z = m->d_z.p; a.forest = m->d_forest.p; a.params = m->d_ptgsk_params.p;
        a.bb0 = 0.98 * 5.670373e-8 * sb_pow4(273.15);
        a.inv_dt_seconds = make_inv_divisor(a.dt_seconds);
        a.inv_dt_us = make_inv_divisor(a.dt_us);
        a.par0 = make_ptgsk_param(m->region_param.data(), param_dt(m));
        a.day_sec_of_year = m->d_doy_soy.p;
        a.ens_params = t.ptgsk_members; a.ens_state_stride = t.state_stride; a.ens_partial_stride = t.partial_stride; a.ens_resp_stride = t.resp_stride;
        for (int k = 0; k < 5; ++k) a.scr[k] = t.scr[k].p;
        a.ens_scr_stride = t.scr_stride;
        // phase pipeline: forcing terms -> snow -> response (sb2_ptgsk.cuh)
        const dim3 ga((unsigned)grid_for(n, SB2_BLOCK_A), (unsigned)grid_for(chunk, SB2_STEPS_A), ne);
        const dim3 gb((unsigned)(grid_for(n, SB2_BLOCK_B) * n_slices), ne), gc((unsigned)(grid_for(n, SB2_BLOCK_C) * n_slices), ne);
        nvtxRangePushA("A forcing_terms");
        if (upar) ptgsk_forcing_terms_kernel<true><<<ga, SB2_BLOCK_A, SB2_MTAB_BYTES, m->stream>>>(a);
        else ptgsk_forcing_terms_kernel<false><<<ga, SB2_BLOCK_A, SB2_MTAB_BYTES, m->stream>>>(a);
        nvtxRangePop();
        zero_tickets();
        nvtxRangePushA("B snow");
        switch (collect & 14) {
#define SB2_CASE(B) case B: if (upar) ptgsk_snow_kernel<B, true><<<gb, SB2_BLOCK_B, SB2_MTAB_BYTES, m->stream>>>(a); \
                            else ptgsk_snow_kernel<B, false><<<gb, SB2_BLOCK_B, SB2_MTAB_BYTES, m->stream>>>(a); break;
            SB2_CASE(0) SB2_CASE(2) SB2_CASE(4) SB2_CASE(6) SB2_CASE(8) SB2_CASE(10) SB2_CASE(12) SB2_CASE(14)
#undef SB2_CASE
        }
        nvtxRangePop();
        zero_tickets();
        nvtxRangePushA("C response");
        switch (collect & 13) {
#define SB2_CASE(B) case B: if (upar) ptgsk_response_kernel<B, true><<<gc, SB2_BLOCK_C, SB2_MTAB_BYTES, m->stream>>>(a); \
                            else ptgsk_response_kernel<B, false><<<gc, SB2_BLOCK_C, SB2_MTAB_BYTES, m->stream>>>(a); break;
            SB2_CASE(0) SB2_CASE(1) SB2_CASE(4) SB2_CASE(5) SB2_CASE(8) SB2_CASE(9) SB2_CASE(12) SB2_CASE(13)
#undef SB2_CASE
        }
        nvtxRangePop();
        m->launches += 3;
    } else {
        const dim3 grid((unsigned)(groups * n_slices), ne);
        zero_tickets();
        if (m->stack == SB2_PT_SS_K) {
            SskRunArgs a{};
            common(a);
            a.params = m->d_ssk_params.p;
            a.inv_dt_hours = make_inv_divisor(a.dt_hours);
            a.step_in_days = a.dt_seconds / 86400.0;
            a.collect = collect & 15;
            ptssk_run_kernel<<<grid, SB2_BLOCK, SB2_MTAB_BYTES, m->stream>>>(a);
        } else if (m->stack == SB2_PT_HPS_K) {
            HpsRunArgs a{};
            common(a);
            a.params = m->d_hps_params.p;
            a.bb0 = 0.98 * 5.670373e-8 * sb_pow4(273.15);  // calculator::BB0 (hbv_physical_snow.h:208)
            a.inv_dt_seconds = make_inv_divisor(a.dt_seconds);
            a.ens_params = t.hps_members; a.ens_state_stride = t.state_stride; a.ens_partial_stride = t.partial_stride; a.ens_resp_stride = t.resp_stride;
            a.collect = collect & 15;
            if (t.hps_members) pthpsk_run_kernel<true><<<grid, SB2_BLOCK, SB2_MTAB_BYTES, m->stream>>>(a);
            else pthpsk_run_kernel<false><<<grid, SB2_BLOCK, SB2_MTAB_BYTES, m->stream>>>(a);
        } else {
            HbvRunArgs a{};
            common(a);
            a.params = m->d_hbv_params.p;
            a.inv_dt_hours = make_inv_divisor(a.dt_hours);
            a.step_in_days = a.dt_seconds / 86400.0;
            a.par0 = make_hbv_param(m->stack == SB2_HBV_STACK, m->region_param.data());
            a.ens_params = t.hbv_members; a.ens_state_stride = t.state_stride; a.ens_partial_stride = t.partial_stride; a.ens_resp_stride = t.resp_stride;
            a.collect = collect & 15;
            if (m->stack == SB2_PT_HS_K) {
                if (upar) hbv_run_kernel<false, true><<<grid, SB2_BLOCK, SB2_MTAB_BYTES, m->stream>>>(a);
                else hbv_run_kernel<false, false><<<grid, SB2_BLOCK, SB2_MTAB_BYTES, m->stream>>>(a);
            } else {
                if (upar) hbv_run_kernel<true, true><<<grid, SB2_BLOCK, SB2_MTAB_BYTES, m->stream>>>(a);
                else hbv_run_kernel<true, false><<<grid, SB2_BLOCK, SB2_MTAB_BYTES, m->stream>>>(a);
            }
        }
        ++m->launches;
    }
    CUDA_OK(cudaGetLastError());
    NvtxRange nv_reduce("catchment_reduce");
    const int64_t total = int64_t(chunk) * m->n_catch();
    catchment_reduce_kernel<<<dim3((unsigned)grid_for(total, 256), ne), 256, 0, m->stream>>>(
        t.partial, m->n_slots, m->d_cat_ptr.p, m->d_cat_slots.p, int(m->n_catch()), chunk, t.cq, t.cc, s0, t.partial_stride, t.catch_stride);
    CUDA_OK(cudaGetLastError());
    ++m->launches;
}

// ---- the cell step over [first, first+n_steps) with forcing/series windows already in place -------------------
void launch_step_range(sb2_model* m, int64_t first, int64_t n_steps, bool collect_end_state) {
    sync_parameters(m);
    sync_filter(m);
    const int64_t n = m->n;
    if (m->partial_steps == 0) {
        // Steps per launch: at most 4 096, and the scratch within 16 GB (measured on 100 000 cells: chunks of 512 / 1 024 / 2 048 / 4 096
        // steps -> 9.23 / 9.42 / 9.54 / 9.62 G cell-steps/s: every launch ends with a tail of one time slice).
        constexpr int64_t cap = 4096, scratch_gb = 16;
        // the per-slot partial sums [ps][n_slots][2] within cap / 4 MB (1 GB at the default)
        int64_t ps = std::max<int64_t>(1, std::min<int64_t>(cap, (int64_t(cap / 4) << 20) / std::max<int64_t>(1, m->n_slots * 16)));
        // pt_gs_k: the five scratch arrays of the phase pipeline are [ps][n] too
        if (m->stack == SB2_PT_GS_K) ps = std::max<int64_t>(16, std::min<int64_t>(ps, (scratch_gb << 30) / (40 * std::max<int64_t>(1, n))));
        m->partial_steps = int(ps);
        m->d_partial.resize(size_t(ps) * m->n_slots * 2);
    }
    if (m->stack == SB2_PT_GS_K)
        for (auto& b : m->d_scr) b.ensure(size_t(std::min<int64_t>(m->partial_steps, n_steps)) * n);
    m->d_tickets.ensure(size_t(1 + step_groups(m)));
    StepTarget t;
    t.state = m->d_state.p; t.partial = m->d_partial.p; t.cq = m->d_cq.p; t.cc = m->d_cc.p; t.scr = m->d_scr;
    t.tickets = m->d_tickets.p;
    t.series = true;
    // chunks of equal length (a whole number of time slices each) rather than full ones and a remainder
    const int64_t n_chunks = std::max<int64_t>(1, (n_steps + m->partial_steps - 1) / m->partial_steps);
    int64_t even = (n_steps + n_chunks - 1) / n_chunks;
    even = std::min<int64_t>(m->partial_steps, (even + 127) / 128 * 128);
    for (int64_t done = 0; done < n_steps; done += even) {
        const int chunk = int(std::min<int64_t>(even, n_steps - done));
        launch_step_chunk(m, t, first + done, chunk, collect_end_state && done + chunk >= n_steps);
    }
}

void check_device_errors(sb2_model* m) {
    int flag = 0;
    CUDA_OK(cudaMemcpyAsync(&flag, m->d_error_flag.p, sizeof(int), cudaMemcpyDeviceToHost, m->stream));
    CUDA_OK(cudaStreamSynchronize(m->stream));
    if (flag) {
        CUDA_OK(cudaMemsetAsync(m->d_error_flag.p, 0, sizeof(int), m->stream));
        if (flag & ERR_KIRCHNER_STEP) throw Error("Max number of iterations exceeded (500). A new step size was not found.");
        if (flag & ERR_HBV_NEGATIVE_OUTFLOW) throw Error("hbv_snow: Negative outflow");
        if (flag & ERR_SKAUGEN_SEARCH) throw Error("skaugen: sca_rel_red found no root (boost::math::tools::bisect: no change of sign) or the gamma density overflowed");
        throw Error("device error flag " + std::to_string(flag));
    }
}

// run_cells argument validation, messages as core/region_model.h:586-592
void validate_run_args(const sb2_model* m, int start_step, int n_steps) {
    if (!(m->T > 0)) throw Error("region_model::run with invalid time_axis invoked");
    if (start_step < 0 || int64_t(start_step) + 1 > m->T) throw Error("region_model::run start_step must in range[0..n_steps-1>");
    if (n_steps < 0) throw Error("region_model::run n_steps must be range[0..time-axis-steps]");
    if (int64_t(start_step) + n_steps > m->T) throw Error("region_model::run start_step+n_steps must be within time-axis range");
}
void snapshot_initial_state_if_unset(sb2_model* m) {
    if (m->has_initial) return;
    m->d_initial_state.resize(m->d_state.n);
    CUDA_OK(cudaMemcpyAsync(m->d_initial_state.p, m->d_state.p, m->d_state.n * sizeof(double), cudaMemcpyDeviceToDevice, m->stream));
    m->has_initial = true;
}

// ---- interpolation ----------------------------------------------------------------------------------------------
IdwParam to_idw(const sb2_idw_parameter& q) {
    IdwParam p{};
    p.max_members = int(q.max_members);
    p.max_distance = q.max_distance;
    p.distance_measure_factor = q.distance_measure_factor;
    p.zscale = q.zscale;
    p.default_temp_gradient = q.default_temp_gradient;
    p.scale_factor = q.scale_factor;
    p.gradient_by_equation = q.gradient_by_equation;
    return p;
}
const sb2_idw_parameter& idw_parameter_of(const sb2_interpolation_parameter& ip, int var) {
    switch (var) {
        case SB2_TEMPERATURE: return ip.temperature_idw;
        case SB2_PRECIPITATION: return ip.precipitation;
        case SB2_RADIATION: return ip.radiation;
        case SB2_WIND_SPEED: return ip.wind_speed;
        default: return ip.rel_hum;
    }
}
int idw_kind_of(int var) {
    switch (var) {
        case SB2_TEMPERATURE: return IDW_TEMPERATURE;
        case SB2_PRECIPITATION: return IDW_PRECIPITATION;
        case SB2_RADIATION: return IDW_RADIATION;
        case SB2_WIND_SPEED: return IDW_WIND_SPEED;
        default: return IDW_REL_HUM;
    }
}

void build_idw_plan(sb2_model* m, int var) {
    IdwPlan& pl = m->idw[var];
    const Source& s = m->src[var];
    pl.p = to_idw(idw_parameter_of(m->ip, var));
    if (pl.p.max_members < 1) throw Error("inverse_distance: max_members must be >= 1");
    pl.n_src = s.n_src;
    const size_t k = size_t(std::min<int64_t>(pl.p.max_members, s.n_src));
    pl.idx.resize(k * m->n); pl.w.resize(k * m->n); pl.f.resize(k * m->n); pl.cnt.resize(m->n);
    // min_weight = 1/distance_measure(origin, (max_distance,0,0)) (inverse_distance.h:160-162)
    const double d2 = pl.p.max_distance * pl.p.max_distance;
    const double min_weight = 1.0 / sb_pow(d2, pl.p.distance_measure_factor / 2.0);
    idw_build_neighbours_kernel<<<grid_for(m->n, 128), 128, 0, m->stream>>>(idw_kind_of(var), m->n, m->d_x.p, m->d_y.p, m->d_z.p, m->d_slope.p,
                                                                           int(s.n_src), s.d_xyz.p, pl.p, min_weight, pl.idx.p, pl.w.p, pl.f.p,
                                                                           pl.cnt.p);
    CUDA_OK(cudaGetLastError());
    ++m->launches;
    pl.valid = true;
    pl.dense_valid = false;
}

int idw_tile_steps(int64_t n_src) {
    const int64_t budget = 32 * 1024 / 8;  // 32 KB of source values per tile
    return int(std::max<int64_t>(1, std::min<int64_t>(64, budget / std::max<int64_t>(1, n_src))));
}

void run_idw(sb2_model* m, int var, int64_t first, int64_t n_steps, double* out) {
    IdwPlan& pl = m->idw[var];
    if (!pl.valid) build_idw_plan(m, var);
    const Source& s = m->src[var];
    if (!s.has_nonfinite && !(var == SB2_TEMPERATURE && pl.p.gradient_by_equation) && s.n_src <= 96 && !m->force_sparse_idw) {
        // every station value is finite: the weighted means are one dense contraction on the FP64 tensor cores
        if (!pl.dense_valid) {
            pl.dense.resize(size_t(s.n_src) * m->n);
            pl.addc.resize(size_t(m->n));
            idw_build_dense_kernel<<<grid_for(m->n, 128), 128, 0, m->stream>>>(idw_kind_of(var), m->n, int(s.n_src), m->d_z.p, pl.p.default_temp_gradient,
                                                                              pl.idx.p, pl.w.p, pl.f.p, pl.cnt.p, pl.dense.p, pl.addc.p);
            CUDA_OK(cudaGetLastError());
            ++m->launches;
            // station compaction lists per tile of the apply kernel (tile shape as dispatched below)
            const int nvp = int(s.n_src);
            const int ks = nvp <= 16 ? 4 : (nvp <= 32 ? 8 : (nvp <= 64 ? 16 : 24)), ntile = nvp <= 32 ? 4 : (nvp <= 64 ? 2 : 1);
            const int64_t n_tiles = grid_for(m->n, 32 * ntile) * 4;  // the apply grid covers whole blocks of four tiles
            pl.ulist.resize(size_t(n_tiles) * ks * 4);
            pl.ukc.resize(size_t(n_tiles));
            CUDA_OK(cudaMemsetAsync(pl.ukc.p, 0, size_t(n_tiles), m->stream));
            idw_union_plan_kernel<<<grid_for(n_tiles * 32, 128), 128, 0, m->stream>>>(m->n, nvp, pl.dense.p, 8 * ntile, ks * 4, pl.ulist.p, pl.ukc.p);
            CUDA_OK(cudaGetLastError());
            ++m->launches;
            std::vector<uint8_t> h_kc(size_t(n_tiles), 0);  // the widest union decides how many k-steps the apply kernel carries
            CUDA_OK(cudaMemcpyAsync(h_kc.data(), pl.ukc.p, h_kc.size(), cudaMemcpyDeviceToHost, m->stream));
            CUDA_OK(cudaStreamSynchronize(m->stream));
            pl.kc_max = 0;
            for (uint8_t k : h_kc) pl.kc_max = std::max(pl.kc_max, int(k));
            pl.dense_valid = true;
        }
        const int nv = int(s.n_src);
        const double* v = s.d_values.p + first * s.n_src;
        const int use_tma = (nv % 2 == 0 && (reinterpret_cast<uintptr_t>(v) & 15) == 0) ? 1 : 0;
#define SB2_DENSE(KS, NT, KROW, TS)                                                                                                       \
    do {                                                                                                                                  \
        const int smem = dense_smem_bytes(KROW, TS);                                                                                      \
        auto kern = dense_apply_dmma_kernel<KS, NT, 0, true, KROW, TS>;                                                                   \
        CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));                                           \
        kern<<<grid_for(m->n, 32 * NT), 128, smem, m->stream>>>(m->n, nullptr, nv, pl.dense.p, pl.addc.p, nullptr, v, s.n_src, nullptr,   \
                                                                int(n_steps), m->d_active.p, out, pl.ulist.p, pl.ukc.p, use_tma,          \
                                                                4 * (nv <= 16 ? 4 : (nv <= 32 ? 8 : (nv <= 64 ? 16 : 24))));              \
    } while (0)
        if (nv <= 16) SB2_DENSE(4, 4, 4, 0);
        else if (nv <= 32) SB2_DENSE(8, 4, 8, 0);
        else if (nv <= 64) {  // rows of 64 stations, k-steps by the widest union of a 16-cell tile
            if (pl.kc_max <= 4) SB2_DENSE(4, 2, 16, SB2_DENSE_TILE_COMPACT);
            else if (pl.kc_max <= 6) SB2_DENSE(6, 2, 16, SB2_DENSE_TILE_COMPACT);
            else if (pl.kc_max <= 8) SB2_DENSE(8, 2, 16, SB2_DENSE_TILE_COMPACT);
            else if (pl.kc_max <= 10) SB2_DENSE(10, 2, 16, SB2_DENSE_TILE_COMPACT);
            else if (pl.kc_max <= 12) SB2_DENSE(12, 2, 16, SB2_DENSE_TILE_COMPACT);
            else SB2_DENSE(16, 2, 16, 0);
        } else SB2_DENSE(24, 1, 24, 0);
#undef SB2_DENSE
        CUDA_OK(cudaGetLastError());
        ++m->launches;
        return;
    }
    const int tile = idw_tile_steps(s.n_src);
    const int max_k = int(std::max<int64_t>(1, std::min<int64_t>(pl.p.max_members, s.n_src)));
    const size_t smem = size_t(tile) * s.n_src * sizeof(double) + size_t(max_k) * IDW_BLOCK * (2 * sizeof(double) + sizeof(int));
    if (smem > 200 * 1024) throw Error("inverse_distance: too many sources / members for the shared-memory tiles");
    const int g = grid_for(m->n, IDW_BLOCK);
#define SB2_IDW(K)                                                                                                                   \
    {                                                                                                                                \
        if (smem > 48 * 1024) CUDA_OK(cudaFuncSetAttribute(idw_apply_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem))); \
        idw_apply_kernel<K><<<g, IDW_BLOCK, smem, m->stream>>>(m->n, m->d_z.p, int(s.n_src), s.d_xyz.p, s.d_values.p, first, int(n_steps),  \
                                                               pl.p, pl.idx.p, pl.w.p, pl.f.p, pl.cnt.p, m->d_active.p, out, tile, max_k);     \
    }
    switch (idw_kind_of(var)) {
        case IDW_TEMPERATURE: SB2_IDW(IDW_TEMPERATURE) break;
        case IDW_PRECIPITATION: SB2_IDW(IDW_PRECIPITATION) break;
        case IDW_RADIATION: SB2_IDW(IDW_RADIATION) break;
        case IDW_WIND_SPEED: SB2_IDW(IDW_WIND_SPEED) break;
        default: SB2_IDW(IDW_REL_HUM) break;
    }
#undef SB2_IDW
    CUDA_OK(cudaGetLastError());
    ++m->launches;
}

BtkOps* btk_ops_for(sb2_model* m, const std::vector<int>& valid, bool check_rank) {
    for (auto& o : m->btk_cache)
        if (o->valid == valid) return o.get();
    if (m->btk_cache.size() >= 8) m->btk_cache.erase(m->btk_cache.begin() + 1);  // keep the full-set operators at slot 0
    const Source& s = m->src[SB2_TEMPERATURE];
    const sb2_btk_parameter& bp = m->ip.temperature;
    host::BtkStationOps h = host::btk_station_ops(s.xyz, valid, bp.sill, bp.nug, bp.range, bp.zscale, bp.gradient_sd, check_rank);
    auto o = std::make_unique<BtkOps>();
    o->valid = valid;
    const int nv = int(valid.size());
    std::vector<double> sub_xyz(size_t(nv) * 3);
    for (int i = 0; i < nv; ++i)
        for (int c = 0; c < 3; ++c) sub_xyz[3 * i + c] = s.xyz[3 * valid[i] + c];
    DevArray<double> d_sub_xyz, d_Kinv, d_FtKinv, d_M22;
    d_sub_xyz.upload(sub_xyz, m->stream);
    d_Kinv.upload(h.K_inv.a, m->stream);
    d_FtKinv.upload(h.FtKinv.a, m->stream);
    d_M22.upload(h.M22.a, m->stream);
    o->E_beta_w.upload(h.E_beta_w.a, m->stream);
    o->sz.upload(h.z, m->stream);
    std::vector<int32_t> vi(valid.begin(), valid.end());
    o->valid_idx.upload(vi, m->stream);
    o->omega.resize(size_t(nv) * m->n);
    o->bm.resize(size_t(2) * m->n);
    m->d_btk_kbuf.ensure(size_t(nv) * m->n);
    btk_build_operators_kernel<<<grid_for(m->n, 128), 128, 0, m->stream>>>(m->n, m->d_x.p, m->d_y.p, m->d_z.p, nv, d_sub_xyz.p, d_Kinv.p,
                                                                          d_FtKinv.p, d_M22.p, bp.sill - bp.nug, bp.range, bp.zscale,
                                                                          o->omega.p, o->bm.p, m->d_btk_kbuf.p);
    CUDA_OK(cudaGetLastError());
    ++m->launches;
    CUDA_OK(cudaStreamSynchronize(m->stream));  // the temporaries above go out of scope
    m->btk_cache.push_back(std::move(o));
    return m->btk_cache.back().get();
}

void run_btk(sb2_model* m, int64_t first, int64_t n_steps, double* out) {
    const Source& s = m->src[SB2_TEMPERATURE];
    const int S = int(s.n_src);
    std::vector<int> all(S);
    for (int i = 0; i < S; ++i) all[i] = i;
    BtkOps* full = btk_ops_for(m, all, true);  // built (and rank-checked) before the time loop, bayesian_kriging.h:300-316
    // segments of constant valid-station set (:333-381)
    int64_t i = 0;
    while (i < n_steps) {
        std::vector<int> valid;
        if (!s.has_nonfinite) valid = all;
        else {
            const double* v = &s.h_values[size_t(first + i) * S];
            for (int k = 0; k < S; ++k) if (std::isfinite(v[k])) valid.push_back(k);
        }
        if (valid.empty()) throw Error("bayesian kriging temperature: No valid sources for time period, giving up.");
        int64_t j = i + 1;
        if (!s.has_nonfinite) j = n_steps;
        else
            for (; j < n_steps; ++j) {
                const double* v = &s.h_values[size_t(first + j) * S];
                bool same = true;
                size_t q = 0;
                for (int k = 0; k < S && same; ++k) {
                    const bool fin = std::isfinite(v[k]);
                    const bool was = q < valid.size() && valid[q] == k;
                    if (fin != was) same = false;
                    if (was) ++q;
                }
                if (!same) break;
            }
        BtkOps* op = int(valid.size()) == S ? full : btk_ops_for(m, valid, false);
        const int nv = int(valid.size());
        const int64_t seg = j - i;
        m->d_btk_beta.ensure(size_t(seg) * 2);
        m->d_btk_resid.ensure(size_t(seg) * nv);
        btk_step_prepare_kernel<<<grid_for(seg, 128), 128, 0, m->stream>>>(int(seg), first + i, S, s.d_values.p, op->valid_idx.p, nv,
                                                                          op->E_beta_w.p, op->sz.p, m->d_btk_beta.p, m->d_btk_resid.p);
        CUDA_OK(cudaGetLastError());
        double* o = out + i * m->n;
        const double* pri = m->d_prior_gradient.p + first + i;
        const int use_tma = (nv % 2 == 0 && (reinterpret_cast<uintptr_t>(m->d_btk_resid.p) & 15) == 0) ? 1 : 0;
#define SB2_BTK(KS, NT, TS)                                                                                                               \
    do {                                                                                                                                  \
        const int smem = dense_smem_bytes(KS, TS);                                                                                        \
        auto kern = dense_apply_dmma_kernel<KS, NT, 1, false, KS, TS>;                                                                    \
        CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));                                           \
        kern<<<grid_for(m->n, 32 * NT), 128, smem, m->stream>>>(m->n, m->d_z.p, nv, op->omega.p, op->bm.p, m->d_btk_beta.p,               \
                                                                m->d_btk_resid.p, nv, pri, int(seg), m->d_active.p, o, nullptr, nullptr,  \
                                                                use_tma, 0);                                                              \
    } while (0)
        if (nv <= 16) SB2_BTK(4, 4, 0);
        else if (nv <= 32) SB2_BTK(8, 4, 0);
        else if (nv <= 64) SB2_BTK(16, 2, 0);
        else if (nv <= 96) SB2_BTK(24, 1, 0);
        else {  // more stations than the register-resident operator tile holds: one thread per cell, operator rows streamed
            const int tile = idw_tile_steps(nv);
            const size_t smem = size_t(tile) * nv * sizeof(double);
            btk_apply_kernel<<<grid_for(m->n, 128), 128, smem, m->stream>>>(m->n, m->d_z.p, nv, op->omega.p, op->bm.p, m->d_btk_beta.p,
                                                                           m->d_btk_resid.p, pri, int(seg), m->d_active.p, o, tile);
        }
#undef SB2_BTK
        CUDA_OK(cudaGetLastError());
        m->launches += 2;
        i = j;
    }
}

// One variable over [first, first+n_steps) into out[(i)*n + c]; the case analysis of region_model.h:456-515
void interpolate_variable(sb2_model* m, int var, int64_t first, int64_t n_steps, double* out) {
    const Source& s = m->src[var];
    if (s.n_src == 0) return;  // env.<var> == nullptr: the cell series keep their NaN fill
    if (var == SB2_TEMPERATURE) {
        if (s.n_src > 1) {
            if (m->ip.use_idw_for_temperature) run_idw(m, var, first, n_steps, out);
            else run_btk(m, first, n_steps, out);
        } else {
            broadcast_source_kernel<<<grid_for(m->n, 128), 128, 0, m->stream>>>(m->n, s.d_values.p + first, int(n_steps), m->d_active.p, out);
            CUDA_OK(cudaGetLastError());
            ++m->launches;
        }
    } else run_idw(m, var, first, n_steps, out);
}

bool interpolate_range(sb2_model* m, int64_t first, int64_t n_steps, int best_effort) {
    NvtxRange nv("interpolate");
    sync_filter(m);
    bool all_ok = true;
    for (int var = 0; var < SB2_N_FORCING; ++var) {
        try {
            interpolate_variable(m, var, first, n_steps, m->d_forcing[var].p + (first - m->forcing_first) * m->n);
        } catch (const std::exception&) {
            if (!best_effort) throw;
            all_ok = false;
        }
    }
    return all_ok;
}

void set_interpolation_parameter(sb2_model* m, const sb2_interpolation_parameter* ip) {
    if (!ip) throw Error("null interpolation parameter");
    if (m->ip_valid && std::memcmp(&m->ip, ip, sizeof(*ip)) == 0) return;
    m->ip = *ip;
    m->ip_valid = true;
    for (auto& pl : m->idw) pl.valid = false;
    m->btk_cache.clear();
}

void ensure_forcing(sb2_model* m, int64_t first, int64_t rows, bool nan_fill) {
    if (m->forcing_first == first && m->forcing_rows == rows && m->d_forcing[0].p) return;
    for (auto& f : m->d_forcing) f.resize(size_t(rows) * m->n);
    m->forcing_first = first;
    m->forcing_rows = rows;
    if (nan_fill)
        for (auto& f : m->d_forcing) fill_nan(m, f.p, rows * m->n);
}

void copy_out_2d(sb2_model* m, const double* d_src /* [rows][n] */, int64_t rows, double* out, int layout) {
    if (layout == SB2_TIME_MAJOR) {
        CUDA_OK(cudaMemcpyAsync(out, d_src, size_t(rows) * m->n * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
    } else {
        DevArray<double> tmp;
        tmp.resize(size_t(rows) * m->n);
        dim3 b(32, 8), g((unsigned)((m->n + 31) / 32), (unsigned)((rows + 31) / 32));
        transpose_kernel<<<g, b, 0, m->stream>>>(d_src, tmp.p, rows, m->n);
        CUDA_OK(cudaGetLastError());
        ++m->launches;
        CUDA_OK(cudaMemcpyAsync(out, tmp.p, size_t(rows) * m->n * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
        CUDA_OK(cudaStreamSynchronize(m->stream));
        return;
    }
    CUDA_OK(cudaStreamSynchronize(m->stream));
}

void time_begin(sb2_model* m, int which) { CUDA_OK(cudaEventRecord(m->ev[which], m->stream)); }
float time_end(sb2_model* m, int a, int b) {
    CUDA_OK(cudaEventRecord(m->ev[b], m->stream));
    CUDA_OK(cudaEventSynchronize(m->ev[b]));
    float ms = 0.f;
    CUDA_OK(cudaEventElapsedTime(&ms, m->ev[a], m->ev[b]));
    return ms;
}
// ---- routing plan (core/routing.h:326-383) ---------------------------------------------------------------------------------
void ensure_routing_plan(sb2_model* m) {
    if (m->route) return;
    if (m->rivers.empty()) throw Error("routing: the river network is empty");
    // routing velocity/alpha/beta live in the cell's parameter set (pt_gs_k.h:102-104, pt_hs_k.h:81-83, hbv_stack.h:93-95)
    const int off = kStacks[m->stack].routing_velocity;
    std::vector<double> cell_routing(size_t(m->n) * 5);
    for (int64_t i = 0; i < m->n; ++i) {
        auto f = m->catch_param.find(m->geo[i].catchment_id);
        const std::vector<double>& p = f != m->catch_param.end() ? f->second : m->region_param;
        double* cr = &cell_routing[5 * i];
        cr[0] = double(m->geo[i].routing_id); cr[1] = m->geo[i].routing_distance;
        cr[2] = p[off]; cr[3] = p[off + 1]; cr[4] = p[off + 2];
    }
    m->route = build_routing_plan(m->rivers, cell_routing, m->n, m->dt, m->stream);
}


// ---- calibration goal function (core/model_calibration.h:830-899) ---------------------------------------------------------
void build_goal_targets(sb2_model* m, std::vector<GoalTarget>& gt, const double* cq, const double* cc, int64_t ens_stride) {
    gt.clear();
    // optimizer::run hands ONE cache vector (catchment_d) to both compute_discharge_sum and compute_charge_sum
    // (model_calibration.h:837,843,855) and each fills it only when empty: whichever of the DISCHARGE / CELL_CHARGE targets comes
    // first in the list decides the series all of them are compared with.  Kept as the reference behaves.
    int first_kind = -1;
    for (auto& tp : m->targets)
        if (first_kind < 0 && (tp->property == SB2_TARGET_DISCHARGE || tp->property == SB2_TARGET_CELL_CHARGE)) first_kind = tp->property;
    for (auto& tp : m->targets) {
        sb2_model::Target& t = *tp;
        GoalTarget g{};
        g.obs = t.d_obs.p;
        g.first_step = (t.t0 - m->t0) / m->dt;
        g.steps_per_period = int32_t(t.dt / m->dt);
        g.n = int32_t(t.obs.size());
        g.calc_mode = (t.calc_mode == SB2_GOAL_ABS_DIFF && t.property == SB2_TARGET_CELL_CHARGE) ? GOAL_ABS_DIFF_SCALED : t.calc_mode;  // :870-873
        g.s_r = t.s_r; g.s_a = t.s_a; g.s_b = t.s_b;
        g.dt_seconds = double(m->dt) / 1e6;
        g.rows = m->T;
        g.scale = nullptr;
        if (t.property == SB2_TARGET_DISCHARGE || t.property == SB2_TARGET_CELL_CHARGE) {
            g.series = first_kind == SB2_TARGET_DISCHARGE ? cq : cc;
            g.ens_stride = ens_stride;
            g.n_col = int32_t(m->n_catch());
            g.cix = t.d_cix.p;
            g.n_cix = int32_t(t.cids.size());
        } else {  // a per-target series [T][1] prepared by the caller
            g.series = t.d_series.p;
            g.ens_stride = 0;
            g.n_col = 1;
            g.cix = t.d_cix.p;  // holds a single 0
            g.n_cix = 1;
        }
        if (!t.aligned) {  // project the property onto the target axis first (single evaluation only; the batch path asks for aligned axes)
            if (ens_stride != 0) throw Error("target_specification: batched evaluation needs target axes aligned with the model axis");
            const int64_t T = m->T, n = int64_t(t.obs.size());
            if (!m->d_axis_t.p || int64_t(m->d_axis_t.n) != T) {
                std::vector<int64_t> tt(static_cast<size_t>(T), 0);
                for (int64_t i = 0; i < T; ++i) tt[size_t(i)] = m->t0 + i * m->dt;
                m->d_axis_t.upload(tt, m->stream);
            }
            DevArray<double> d_prop, d_a, d_b;
            d_prop.resize(size_t(T));
            t.d_projected.resize(size_t(n));
            auto project = [&](int mode, double* out) {
                goal_property_kernel<<<grid_for(T, 256), 256, 0, m->stream>>>(g.series, T, g.n_col, g.cix, g.n_cix, mode, d_prop.p);
                if (t.points.empty())
                    average_accessor_kernel<<<grid_for(n, 256), 256, 0, m->stream>>>(m->d_axis_t.p, d_prop.p, T, 1, m->t0 + T * m->dt, 0, t.t0, t.dt, n, out);
                else
                    average_accessor_periods_kernel<<<grid_for(n, 256), 256, 0, m->stream>>>(m->d_axis_t.p, d_prop.p, T, m->t0 + T * m->dt, 0,
                                                                                            t.d_points.p, n, out);
                CUDA_OK(cudaGetLastError());
                m->launches += 2;
            };
            project(0, t.d_projected.p);
            if (g.calc_mode == GOAL_ABS_DIFF_SCALED) {
                d_a.resize(size_t(n)); d_b.resize(size_t(n));
                t.d_scale.resize(size_t(n));
                project(1, d_a.p);
                project(2, d_b.p);
                goal_max_kernel<<<grid_for(n, 256), 256, 0, m->stream>>>(d_a.p, d_b.p, n, t.d_scale.p);
                CUDA_OK(cudaGetLastError());
                ++m->launches;
                g.scale = t.d_scale.p;
            }
            CUDA_OK(cudaStreamSynchronize(m->stream));  // the temporaries go out of scope
            m->d_one_zero.ensure(1);
            CUDA_OK(cudaMemsetAsync(m->d_one_zero.p, 0, sizeof(int32_t), m->stream));
            g.series = t.d_projected.p; g.ens_stride = 0; g.n_col = 1; g.cix = m->d_one_zero.p; g.n_cix = 1;
            g.first_step = 0; g.steps_per_period = 1; g.rows = n;
            g.dt_seconds = 1.0;  // (v * 1) / 1 = v: the projected value is taken as it is
        }
        gt.push_back(g);
    }
}

// weighted mean over the targets with a finite partial value (:881-887)
double combine_goal(const sb2_model* m, const double* partial) {
    double goal = 0.0, scale_sum = 0.0;
    for (size_t k = 0; k < m->targets.size(); ++k)
        if (std::isfinite(partial[k])) { scale_sum += m->targets[k]->scale_factor; goal += m->targets[k]->scale_factor * partial[k]; }
    return goal / scale_sum;
}

void prepare_snow_and_routed_targets(sb2_model* m) {
    for (auto& tp : m->targets) {
        sb2_model::Target& t = *tp;
        if (t.property == SB2_TARGET_SNOW_COVERED_AREA || t.property == SB2_TARGET_SNOW_WATER_EQUIVALENT) {
            const int r = t.property == SB2_TARGET_SNOW_COVERED_AREA ? SB2_R_SNOW_SCA : SB2_R_SNOW_SWE;
            if (!m->d_resp[r].p || m->out_first != 0 || m->out_rows != m->T) throw Error(r == SB2_R_SNOW_SCA ? "resource collector doesn't have snow_sca" : "resource collector doesn't have snow_swe");
            // area-weighted mean over all cells of the target's catchments (:765-790)
            std::vector<int32_t> cells;
            for (int64_t i = 0; i < m->n; ++i)
                for (auto cid : t.cids)
                    if (m->geo[i].catchment_id == cid) { cells.push_back(int32_t(i)); break; }
            std::vector<int32_t> ptr{0, int32_t(cells.size())};
            DevArray<int32_t> d_ptr, d_cells;
            d_ptr.upload(ptr, m->stream);
            d_cells.upload(cells, m->stream);
            t.d_series.resize(size_t(m->T));
            catchment_area_mean_kernel<<<grid_for(m->T, 256), 256, 0, m->stream>>>(m->d_resp[r].p, m->d_area.p, d_ptr.p, d_cells.p, 1, m->T, m->n,
                                                                                  t.d_series.p);
            CUDA_OK(cudaGetLastError());
            ++m->launches;
            CUDA_OK(cudaStreamSynchronize(m->stream));
        } else if (t.property == SB2_TARGET_ROUTED_DISCHARGE) {
            std::vector<double> out(size_t(m->T));
            if (sb2_river_flows(m, t.river_id, 0, m->T, nullptr, nullptr, out.data()) != 0) throw Error(m->err);
            t.d_series.upload(out, m->stream);
            CUDA_OK(cudaStreamSynchronize(m->stream));
        }
    }
}

double evaluate_goal_single(sb2_model* m) {
    prepare_snow_and_routed_targets(m);
    std::vector<GoalTarget> gt;
    build_goal_targets(m, gt, m->d_cq.p, m->d_cc.p, 0);
    DevArray<GoalTarget> d_gt;
    DevArray<double> d_out;
    d_gt.upload(gt, m->stream);
    d_out.resize(gt.size());
    goal_kernel<<<dim3((unsigned)gt.size(), 1), 256, 0, m->stream>>>(d_gt.p, int(gt.size()), d_out.p);
    CUDA_OK(cudaGetLastError());
    ++m->launches;
    std::vector<double> partial(gt.size());
    CUDA_OK(cudaMemcpyAsync(partial.data(), d_out.p, partial.size() * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
    CUDA_OK(cudaStreamSynchronize(m->stream));
    return combine_goal(m, partial.data());
}

// the longest cell unit hydrograph (routing.h:119-123) any of the n_sets parameter sets gives a routed cell, cells under a catchment
// override with the override's velocity: a routed batch carries this minus one rows of cell discharge from one chunk of steps to the
// next.  uhg_steps is monotone in the distance, so for a member's own cells the shortest and the longest distance decide it.
int64_t batch_cell_uhg_max_len(const sb2_model* m, int64_t n_sets, const double* P) {
    const int off = kStacks[m->stack].routing_velocity;
    auto len = [&](double distance, double velocity) { return std::max<int64_t>(1, host::uhg_steps(distance, velocity, m->dt)); };
    int64_t max_len = 1;
    double dmin = INFINITY, dmax = -INFINITY;
    for (int64_t i = 0; i < m->n; ++i) {
        if (m->geo[i].routing_id <= 0) continue;
        auto f = m->catch_param.find(m->geo[i].catchment_id);
        if (f != m->catch_param.end()) max_len = std::max(max_len, len(m->geo[i].routing_distance, f->second[off]));
        else { dmin = std::min(dmin, m->geo[i].routing_distance); dmax = std::max(dmax, m->geo[i].routing_distance); }
    }
    if (dmin <= dmax)
        for (int64_t e = 0; e < n_sets; ++e) {
            const double v = P[e * m->n_param + off];
            max_len = std::max(max_len, std::max(len(dmin, v), len(dmax, v)));
        }
    return max_len;
}

// ensemble of region-parameter sets for pt_gs_k, pt_hs_k, hbv_stack and pt_hps_k: member e = one grid layer of the step kernels
// run_cells launches, stepping its own copy of the state; the model's parameters, state, catchment series and river flows are left
// as they are.  A ROUTED_DISCHARGE target routes every member as sb2_river_flows routes a run: each chunk's cell discharge goes through
// the local-inflow kernel with the previous chunks' last H rows in front of it (as run_windowed does per window), then the river
// network is routed level by level, all members in one launch each, with the member's own cell unit hydrographs.
void goal_batch(sb2_model* m, int64_t n_sets, const double* P, double* goals) {
    sync_parameters(m);
    sync_filter(m);
    const bool gsk = m->stack == SB2_PT_GS_K;
    const int64_t n = m->n, T = m->T, nc = m->n_catch();
    const size_t state_sz = size_t(m->n_state) * n;
    bool routed = false;
    for (auto& tp : m->targets) routed = routed || tp->property == SB2_TARGET_ROUTED_DISCHARGE;
    if (routed && m->rivers.empty()) throw Error("routing: the river network is empty");
    const int64_t n_riv = int64_t(m->rivers.size() / 6);
    const int64_t H = routed ? batch_cell_uhg_max_len(m, n_sets, P) - 1 : 0;
    // members per pass from a ~12 GB budget: state + catchment series (discharge, charge); with a routed target also the river series
    // (local inflow, upstream inflow, output: [n_riv][T] each) and the H history rows of the two cell-discharge buffers below
    size_t per_member = state_sz * 8 + size_t(T) * nc * 16;
    if (routed) per_member += size_t(3) * n_riv * T * 8 + size_t(2) * H * n * 8;
    const int64_t E = std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(n_sets, 65535), int64_t((12ULL << 30) / per_member)));
    // steps per pass: ~1 GB of per-slot partial sums; pt_gs_k also ~4 GB of phase-pipeline scratch (five [E][ps][n] arrays); a routed
    // target ~2 GB for the step rows of the two cell-discharge buffers ([E][H + ps][n] each)
    int64_t ps = std::min<int64_t>(T, int64_t((1ULL << 30) / (size_t(E) * m->n_slots * 16)));
    if (gsk) ps = std::min<int64_t>(ps, std::max<int64_t>(8, int64_t((4ULL << 30) / (size_t(E) * n * 40))));
    if (routed) ps = std::min<int64_t>(ps, int64_t((2ULL << 30) / (size_t(E) * n * 16)));
    ps = std::max<int64_t>(1, ps);
    DevArray<double> d_state, d_partial, d_cq, d_cc, d_out, d_scr[5];
    if (gsk)
        for (auto& b : d_scr) b.resize(size_t(E) * ps * n);
    DevArray<int> d_tickets;
    d_tickets.resize(size_t(E) * (1 + step_groups(m)));
    DevArray<PtgskParam> d_par;
    DevArray<HbvParam> d_hbv_par;
    DevArray<HpsParam> d_hps_par;
    DevArray<GoalTarget> d_gt;
    d_state.resize(size_t(E) * state_sz);
    d_partial.resize(size_t(E) * ps * m->n_slots * 2);
    d_cq.resize(size_t(E) * T * nc);
    d_cc.resize(size_t(E) * T * nc);
    d_out.resize(size_t(E) * m->targets.size());
    // routed: a pair of [E][H + ps][n] cell-discharge buffers.  A chunk's steps write buffer `cur` from row H on, after the history
    // rows; its last H rows are then copied to the front of the other buffer, which the next chunk writes.  The members' cell charge,
    // needed by nothing here, goes to the other buffer's step rows, which the next chunk overwrites.  Cells outside the calculation
    // filter are never written and read NaN, as in the NaN-initialised series of run_cells.
    const int64_t qrows = H + ps;
    DevArray<double> d_qbuf[2], d_rlocal, d_rup, d_rout;
    if (routed) {
        for (auto& b : d_qbuf) { b.resize(size_t(E) * qrows * n); fill_nan(m, b.p, E * qrows * n); }
        d_rlocal.resize(size_t(E) * n_riv * T);
        d_rup.resize(size_t(E) * n_riv * T);
        d_rout.resize(size_t(E) * n_riv * T);
    }
    std::vector<GoalTarget> gt;
    build_goal_targets(m, gt, d_cq.p, d_cc.p, T * nc);
    std::vector<int64_t> riv_ix(gt.size(), -1);  // a routed target's river: the position in the network table, as in the plan
    for (size_t k = 0; k < gt.size(); ++k) {
        if (m->targets[k]->property != SB2_TARGET_ROUTED_DISCHARGE) continue;
        for (int64_t r = 0; r < n_riv; ++r)
            if (int64_t(m->rivers[6 * r]) == m->targets[k]->river_id) riv_ix[k] = r;
        if (riv_ix[k] >= 0) { gt[k].series = d_rout.p + riv_ix[k] * T; gt[k].ens_stride = n_riv * T; }
    }
    d_gt.upload(gt, m->stream);
    StepTarget t;
    t.state = d_state.p; t.partial = d_partial.p; t.cq = d_cq.p; t.cc = d_cc.p; t.scr = d_scr;
    t.state_stride = int64_t(state_sz); t.partial_stride = ps * m->n_slots * 2; t.catch_stride = T * nc; t.scr_stride = ps * n;
    t.tickets = d_tickets.p;
    t.resp_stride = qrows * n;
    std::vector<double> partial(size_t(E) * gt.size());
    for (int64_t e0 = 0; e0 < n_sets; e0 += E) {
        const int64_t ne = std::min<int64_t>(E, n_sets - e0);
        std::vector<const double*> sets;
        for (int64_t e = 0; e < ne; ++e) sets.push_back(P + (e0 + e) * m->n_param);
        if (gsk) { upload_params(m, sets, d_par); t.ptgsk_members = d_par.p; }
        else if (m->stack == SB2_PT_HPS_K) { upload_params(m, sets, d_hps_par); t.hps_members = d_hps_par.p; }
        else { upload_params(m, sets, d_hbv_par); t.hbv_members = d_hbv_par.p; }
        t.members = int(ne);
        std::unique_ptr<RoutingPlan> route;
        if (routed) {  // the cells' routing triples as ensure_routing_plan takes them, member by member
            const int off = kStacks[m->stack].routing_velocity;
            std::vector<double> cell_routing(size_t(ne) * n * 5);
            for (int64_t e = 0; e < ne; ++e)
                for (int64_t i = 0; i < n; ++i) {
                    auto f = m->catch_param.find(m->geo[i].catchment_id);
                    const double* p = f != m->catch_param.end() ? f->second.data() : sets[size_t(e)];
                    double* cr = &cell_routing[(size_t(e) * n + i) * 5];
                    cr[0] = double(m->geo[i].routing_id); cr[1] = m->geo[i].routing_distance;
                    cr[2] = p[off]; cr[3] = p[off + 1]; cr[4] = p[off + 2];
                }
            route = build_routing_plan(m->rivers, cell_routing, n, m->dt, m->stream);
            for (size_t k = 0; k < gt.size(); ++k)  // sb2_river_flows' checks, in its order
                if (m->targets[k]->property == SB2_TARGET_ROUTED_DISCHARGE && riv_ix[k] < 0)
                    throw Error("river network: river id " + std::to_string(m->targets[k]->river_id) + " not found");
            if (!(m->collect_bits & SB2_COLLECT_DISCHARGE))
                throw Error("river flows need avg_discharge over the whole time axis (run_cells with a discharge collector, or run_windowed with the river network set)");
            if (route->cell_max_len - 1 > H) throw Error("routing: cell unit hydrograph longer than the batch's history");
        }
        for (int64_t e = 0; e < ne; ++e)  // reset_states(): every member starts from the initial state (:833)
            CUDA_OK(cudaMemcpyAsync(d_state.p + e * state_sz, m->d_initial_state.p, state_sz * sizeof(double), cudaMemcpyDeviceToDevice, m->stream));
        int cur = 0;
        for (int64_t done = 0; done < T; done += ps) {
            const int chunk = int(std::min<int64_t>(ps, T - done));
            if (routed) { t.q = d_qbuf[cur].p + H * n; t.charge = d_qbuf[cur ^ 1].p + H * n; }
            launch_step_chunk(m, t, done, chunk, false);
            if (routed) {
                routing_local_inflow(*route, t.q, n, chunk, H, done, T, d_rlocal.p, m->stream, &m->launches, int(ne), qrows * n);
                if (H > 0 && done + chunk < T) {
                    route_history_kernel<<<dim3((unsigned)std::min<int64_t>(grid_for(H * n, 256), 1024), (unsigned)ne), 256, 0, m->stream>>>(
                        d_qbuf[cur].p, d_qbuf[cur ^ 1].p, qrows * n, int64_t(chunk) * n, H * n);
                    CUDA_OK(cudaGetLastError());
                    ++m->launches;
                }
                cur ^= 1;
            }
        }
        if (routed) routing_network(*route, T, d_rlocal.p, d_rup.p, d_rout.p, m->stream, &m->launches, int(ne));
        goal_kernel<<<dim3((unsigned)gt.size(), (unsigned)ne), 256, 0, m->stream>>>(d_gt.p, int(gt.size()), d_out.p);
        CUDA_OK(cudaGetLastError());
        ++m->launches;
        CUDA_OK(cudaMemcpyAsync(partial.data(), d_out.p, size_t(ne) * gt.size() * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
        CUDA_OK(cudaStreamSynchronize(m->stream));
        for (int64_t e = 0; e < ne; ++e) goals[e0 + e] = combine_goal(m, partial.data() + e * gt.size());
    }
    check_device_errors(m);
}

// ---- statistics readers (core/cell_model.h:194-406) ------------------------------------------------------------------
// verify_cids_exist (:197-213) + the per-cell selection of is_match (:215-218): a cell is selected once if any index matches
std::vector<uint8_t> stat_selection(const sb2_model* m, const int64_t* indexes, int n_indexes, int scope) {
    if (m->n == 0) throw Error("no cells to make statistics on");
    std::vector<uint8_t> sel(size_t(m->n), n_indexes == 0 ? 1 : 0);
    if (n_indexes == 0) return sel;
    if (!indexes) throw Error("null index list");
    if (scope == SB2_SCOPE_CELL_IX) {
        for (int k = 0; k < n_indexes; ++k) {
            const int64_t cid = indexes[k];
            if (cid < 0 || cid > m->n)
                throw Error("Supplied cell index reference " + std::to_string(cid) + " is ouside valid range 0 .." + std::to_string(m->n));
            if (cid < m->n) sel[size_t(cid)] = 1;
        }
    } else if (scope == SB2_SCOPE_CATCHMENT_IX) {
        std::vector<uint8_t> by_cix(size_t(m->n_catch()), 0);
        for (int k = 0; k < n_indexes; ++k) {
            auto f = m->cid_to_cix.find(indexes[k]);
            if (f == m->cid_to_cix.end()) throw Error("one or more supplied catchment_indexes does not exist:" + std::to_string(indexes[k]));
            by_cix[size_t(f->second)] = 1;
        }
        for (int64_t i = 0; i < m->n; ++i) sel[size_t(i)] = by_cix[size_t(m->cix_of_cell[i])];
    } else
        throw Error("unknown statistics scope");
    return sel;
}
// per-cell ae_scale_factor for the pot_ratio statistic (null for every other series)
const double* stat_ae_scale(sb2_model* m, int kind, DevArray<double>& buf) {
    if (kind != SB2_STAT_AE_POT_RATIO) return nullptr;
    sync_parameters(m);
    buf.resize(size_t(m->n));
    if (m->stack == SB2_PT_GS_K)
        stat_cell_ae_scale_kernel<<<grid_for(m->n, 256), 256, 0, m->stream>>>(m->n, m->d_pset.p, m->d_ptgsk_params.p, buf.p);
    else if (m->stack == SB2_PT_SS_K)
        stat_cell_ae_scale_ssk_kernel<<<grid_for(m->n, 256), 256, 0, m->stream>>>(m->n, m->d_pset.p, m->d_ssk_params.p, buf.p);
    else if (m->stack == SB2_PT_HPS_K)
        stat_cell_ae_scale_hps_kernel<<<grid_for(m->n, 256), 256, 0, m->stream>>>(m->n, m->d_pset.p, m->d_hps_params.p, buf.p);
    else
        stat_cell_ae_scale_hbv_kernel<<<grid_for(m->n, 256), 256, 0, m->stream>>>(m->n, m->d_pset.p, m->d_hbv_params.p, buf.p);
    CUDA_OK(cudaGetLastError());
    ++m->launches;
    return buf.p;
}
// the resident rows of a per-cell series: device pointer of row `start`, after checking [start, start+rows) is resident
const double* stat_series_rows(const sb2_model* m, int kind, int series, int64_t start, int64_t rows) {
    const double* base = nullptr;
    int64_t first = 0, have = 0;
    if (kind == SB2_STAT_AE_POT_RATIO) {
        if (m->stack == SB2_HBV_STACK) throw Error("pot_ratio statistics need a Kirchner stack (pt_gs_k, pt_hs_k)");
        kind = SB2_STAT_STATE;
        series = SB2_S_KIRCHNER_DISCHARGE;
    }
    if (kind == SB2_STAT_FORCING) {
        if (series < 0 || series >= SB2_N_FORCING) throw Error("unknown forcing variable");
        base = m->d_forcing[series].p; first = m->forcing_first; have = m->forcing_rows;
    } else if (kind == SB2_STAT_RESPONSE) {
        if (series < 0 || series >= SB2_N_RESPONSE) throw Error("unknown response series");
        base = m->d_resp[series].p; first = m->out_first; have = m->out_rows;
        if (!base) throw Error("response series is not collected in the current collector mode");
    } else if (kind == SB2_STAT_STATE) {
        if (series < 0 || series >= SB2_N_STATE_SERIES) throw Error("unknown state series");
        base = m->d_st[series].p; first = m->out_first; have = m->out_rows + 1;
        if (!base) throw Error("state series is not collected in the current collector mode");
    } else
        throw Error("unknown statistics series kind");
    if (!base) throw Error("the cell environment is not initialised");
    if (rows < 0 || start < first || start + rows > first + have) throw Error("requested steps are outside the resident series window");
    return base + (start - first) * m->n;
}

}  // namespace

// ====================================================================================================================
extern "C" {

int sb2_version(void) { return 100; }

void sb2_interpolation_parameter_default(sb2_interpolation_parameter* ip) {
    if (!ip) return;
    std::memset(ip, 0, sizeof(*ip));
    ip->temperature = sb2_btk_parameter{0.0025, 25.0, 0.5, 200000.0, 20.0};  // bayesian_kriging.h:204-217
    ip->use_idw_for_temperature = 0;
    auto idw = [](int64_t mm) {
        sb2_idw_parameter p{};
        p.max_members = mm; p.max_distance = 200000.0; p.distance_measure_factor = 2.0; p.zscale = 1.0;
        p.default_temp_gradient = -0.006; p.gradient_by_equation = 0; p.scale_factor = 1.02;
        return p;
    };
    ip->temperature_idw = idw(20);  // inverse_distance.h:56-62
    ip->precipitation = idw(20);    // :70-74
    ip->wind_speed = idw(10);       // :38-48
    ip->radiation = idw(10);
    ip->rel_hum = idw(10);
}

int sb2_model_create(int stack, int64_t n_cells, const sb2_geo_cell* cells, int device, sb2_model** out) {
    if (out) *out = nullptr;
    std::unique_ptr<sb2_model> m;
    try {
        if (!out) throw Error("null output pointer");
        if (stack < 0 || stack > 4) throw Error("unknown method stack");
        if (n_cells <= 0 || !cells) throw Error("region_model needs at least one cell");
        int count = 0;
        cudaError_t e = cudaGetDeviceCount(&count);
        if (e != cudaSuccess || count == 0) {
            cudaGetLastError();
            throw Error(std::string("no CUDA device available (") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count 0") +
                        "); shyft_b200 has no CPU path");
        }
        if (device < 0 || device >= count) throw Error("CUDA device ordinal out of range");
        m.reset(new sb2_model());
        m->stack = stack; m->device = device; m->n = n_cells;
        m->use_device();
        m->geo.assign(cells, cells + n_cells);
        const StackInfo& info = kStacks[stack];
        m->n_param = int(info.parameter.size()); m->n_state = int(info.state.size());
        // update_ix_to_id_mapping (region_model.h:233-249): cix in order of first appearance of the catchment id
        m->cix_of_cell.resize(n_cells);
        for (int64_t i = 0; i < n_cells; ++i) {
            auto f = m->cid_to_cix.find(cells[i].catchment_id);
            if (f == m->cid_to_cix.end()) {
                m->cid_to_cix[cells[i].catchment_id] = int64_t(m->cix_to_cid.size());
                m->cix_of_cell[i] = int64_t(m->cix_to_cid.size());
                m->cix_to_cid.push_back(cells[i].catchment_id);
            } else m->cix_of_cell[i] = f->second;
        }
        std::vector<double> col(n_cells);
        auto up = [&](DevArray<double>& d, auto get) {
            for (int64_t i = 0; i < n_cells; ++i) col[i] = get(cells[i]);
            d.upload(col, m->stream);
            CUDA_OK(cudaStreamSynchronize(m->stream));
        };
        up(m->d_x, [](const sb2_geo_cell& g) { return g.x; });
        up(m->d_y, [](const sb2_geo_cell& g) { return g.y; });
        up(m->d_z, [](const sb2_geo_cell& g) { return g.z; });
        up(m->d_area, [](const sb2_geo_cell& g) { return g.area; });
        up(m->d_glacier, [](const sb2_geo_cell& g) { return g.glacier; });
        up(m->d_lake, [](const sb2_geo_cell& g) { return g.lake; });
        up(m->d_reservoir, [](const sb2_geo_cell& g) { return g.reservoir; });
        up(m->d_forest, [](const sb2_geo_cell& g) { return g.forest; });
        up(m->d_slope, [](const sb2_geo_cell& g) { return g.radiation_slope_factor; });
        m->region_param = info.parameter;
        std::vector<double> soa(size_t(m->n_state) * n_cells);
        for (int s = 0; s < m->n_state; ++s)
            for (int64_t i = 0; i < n_cells; ++i) soa[size_t(s) * n_cells + i] = info.state[s];
        m->d_state.upload(soa, m->stream);
        m->d_error_flag.resize(1);
        CUDA_OK(cudaMemsetAsync(m->d_error_flag.p, 0, sizeof(int), m->stream));
        build_slots(m.get());
        for (auto& ev : m->ev) CUDA_OK(cudaEventCreate(&ev));
        CUDA_OK(cudaStreamSynchronize(m->stream));
        *out = m.release();
        return 0;
    } catch (const std::exception& e) {
        g_create_error = e.what();
        return 1;
    }
}

void sb2_model_destroy(sb2_model* m) {
    if (!m) return;
    cudaSetDevice(m->device);
    cudaStreamSynchronize(m->stream);
    for (auto& ev : m->ev) if (ev) cudaEventDestroy(ev);
    delete m;
}

const char* sb2_last_error(const sb2_model* m) { return m ? m->err.c_str() : g_create_error.c_str(); }

int64_t sb2_size(const sb2_model* m) { return m ? m->n : -1; }
int64_t sb2_number_of_catchments(const sb2_model* m) { return m ? m->n_catch() : -1; }
int sb2_catchment_ids(const sb2_model* m, int64_t* out) {
    return guarded_c(m, [&] { std::copy(m->cix_to_cid.begin(), m->cix_to_cid.end(), out); });
}
int sb2_cell_catchment_ix(const sb2_model* m, int64_t* out) {
    return guarded_c(m, [&] { std::copy(m->cix_of_cell.begin(), m->cix_of_cell.end(), out); });
}
int sb2_parameter_size(const sb2_model* m) { return m ? m->n_param : -1; }
int sb2_state_size(const sb2_model* m) { return m ? m->n_state : -1; }

// ---- parameters, filter, state -------------------------------------------------------------------------------------
int sb2_set_region_parameter(sb2_model* m, const double* p, int n) {
    return guarded(m, [&] {
        if (n != m->n_param) throw Error("parameter vector size does not match parameter::size()");
        m->region_param.assign(p, p + n);
        m->param_dirty = true;
        m->route.reset();  // the cells' unit hydrographs carry the routing velocity / alpha / beta of the parameter set
        m->rlocal_valid = m->rnet_valid = false;
    });
}
int sb2_get_region_parameter(const sb2_model* m, double* p, int n) {
    return guarded_c(m, [&] {
        if (n != m->n_param) throw Error("parameter vector size does not match parameter::size()");
        std::copy(m->region_param.begin(), m->region_param.end(), p);
    });
}
int sb2_set_catchment_parameter(sb2_model* m, int64_t cid, const double* p, int n) {
    return guarded(m, [&] {
        if (n != m->n_param) throw Error("parameter vector size does not match parameter::size()");
        m->catch_param[cid].assign(p, p + n);
        m->param_dirty = true;
        m->route.reset();  // as sb2_remove_catchment_parameter
        m->rlocal_valid = m->rnet_valid = false;
    });
}
int sb2_get_catchment_parameter(const sb2_model* m, int64_t cid, double* p, int n) {
    return guarded_c(m, [&] {
        if (n != m->n_param) throw Error("parameter vector size does not match parameter::size()");
        auto f = m->catch_param.find(cid);
        const std::vector<double>& v = f != m->catch_param.end() ? f->second : m->region_param;
        std::copy(v.begin(), v.end(), p);
    });
}
int sb2_remove_catchment_parameter(sb2_model* m, int64_t cid) {
    return guarded(m, [&] {
        if (m->catch_param.erase(cid)) {
            m->param_dirty = true;
            m->route.reset();  // the cells' unit hydrographs carry the removed override's routing velocity / alpha / beta
            m->rlocal_valid = m->rnet_valid = false;
        }
    });
}
int sb2_has_catchment_parameter(const sb2_model* m, int64_t cid) { return m && m->catch_param.count(cid) ? 1 : 0; }

int sb2_set_catchment_calculation_filter(sb2_model* m, const int64_t* cids, int n) {
    return guarded(m, [&] {
        if (n > 0) {
            if (int64_t(n) > m->n_catch()) throw Error("set_catchment_calculation_filter: supplied list > available catchments");
            for (int i = 0; i < n; ++i)
                if (!m->cid_to_cix.count(cids[i])) throw Error("set_catchment_calculation_filter: no cells have supplied cid");
            m->catchment_filter.assign(m->n_catch(), 0);
            for (int i = 0; i < n; ++i) m->catchment_filter[m->cid_to_cix[cids[i]]] = 1;
        } else m->catchment_filter.clear();
        m->filter_dirty = true;
    });
}

int sb2_set_states(sb2_model* m, const double* states, int64_t n_cells) {
    return guarded(m, [&] {
        if (n_cells != m->n) throw Error("Length of the state vector must equal number of cells");
        std::vector<double> soa(size_t(m->n_state) * m->n);
        for (int64_t i = 0; i < m->n; ++i)
            for (int s = 0; s < m->n_state; ++s) soa[size_t(s) * m->n + i] = states[i * m->n_state + s];
        m->d_state.upload(soa, m->stream);
        CUDA_OK(cudaStreamSynchronize(m->stream));
        if (!m->has_initial) {  // first set_states establishes the initial state (region_model.h:806-808)
            m->d_initial_state.upload(soa, m->stream);
            CUDA_OK(cudaStreamSynchronize(m->stream));
            m->has_initial = true;
        }
    });
}
// hbv_snow::state::distribute(parameter, force = false) (core/hbv_snow.h:114-118 over hbv_snow_common.h:44-67), which pt_hs_k::run and
// run_hbv_stack call first (core/pt_hs_k.h:230, core/hbv_stack.h:312): a state given as (swe, sca) with EMPTY bin vectors -- the usual
// HbvSnowState(swe, sca) -- gets its bins from swe and sca.  The flat state of this ABI always carries the 5 + 5 bins, so "empty" is spelled
// "all ten bins zero": such rows are distributed here (host side, before set_states); rows with any non-zero bin are left alone, exactly as
// a state whose vectors already have the parameter's size.  states: [cell][state_size] in place, n_cells rows in the model's cell order.
int sb2_hbv_distribute_snow(const sb2_model* cm, double* states, int64_t n_cells) {
    return guarded_c(cm, [&] {
        sb2_model* m = const_cast<sb2_model*>(cm);
        if (m->stack == SB2_PT_GS_K || m->stack == SB2_PT_SS_K) throw Error("distribute_snow: this stack's state has no snow bins");
        if (m->stack == SB2_PT_HPS_K) throw Error("distribute_snow: a pt_hps_k state carries its bins (and their albedo / iso_pot_energy) explicitly");
        if (n_cells != m->n) throw Error("Length of the state vector must equal number of cells");
        const int lw_ix = m->stack == SB2_PT_HS_K ? 4 : 8;  // hs.lw in parameter::get order
        for (int64_t i = 0; i < m->n; ++i) {
            double* st = states + i * m->n_state;
            double *swe = st, *sca = st + 1, *sp = st + 2, *sw = st + 2 + HBV_NB;
            bool empty = true;
            for (int k = 0; k < 2 * HBV_NB; ++k) empty = empty && sp[k] == 0.0;
            if (!empty) continue;
            auto f = m->catch_param.find(m->geo[i].catchment_id);
            const std::vector<double>& pv = f != m->catch_param.end() ? f->second : m->region_param;
            const HbvParam p = make_hbv_param(m->stack == SB2_HBV_STACK, pv.data());
            const double lw = pv[lw_ix];
            if (*swe <= 1.0e-3 || *sca <= 1.0e-3) { *swe = *sca = 0.0; continue; }
            for (int k = 0; k < HBV_NB; ++k) sp[k] = *sca < p.I[k] ? 0.0 : p.s[k] * *swe;
            // integrate(sp, intervals, n, 0.0, sca, true), hbv_snow_common.h:14-43 with a = x[0]
            double area = 0.0, f_l = sp[0], x_l = 0.0;
            for (int left = 0; left < HBV_NB - 1; ++left) {
                if (*sca >= p.I[left + 1]) {
                    area += 0.5 * (f_l + sp[left + 1]) * (p.I[left + 1] - x_l);
                    x_l = p.I[left + 1];
                    f_l = sp[left + 1];
                } else {
                    area += 0.5 * f_l * (*sca - x_l);
                    break;
                }
            }
            if (area < *swe) {
                const double corr1 = *swe / area * lw, corr2 = *swe / area * (1.0 - lw);
                for (int k = 0; k < HBV_NB; ++k) { sw[k] = corr1 * sp[k]; sp[k] *= corr2; }
            }
        }
    });
}
int sb2_get_states(const sb2_model* m, double* states, int64_t n_cells) {
    return guarded_c(m, [&] {
        if (n_cells != m->n) throw Error("Length of the state vector must equal number of cells");
        std::vector<double> soa(size_t(m->n_state) * m->n);
        CUDA_OK(cudaMemcpyAsync(soa.data(), m->d_state.p, soa.size() * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
        CUDA_OK(cudaStreamSynchronize(m->stream));
        for (int64_t i = 0; i < m->n; ++i)
            for (int s = 0; s < m->n_state; ++s) states[i * m->n_state + s] = soa[size_t(s) * m->n + i];
    });
}
int sb2_set_initial_state(sb2_model* m, const double* states, int64_t n_cells) {
    return guarded(m, [&] {
        if (n_cells != m->n) throw Error("Length of the state vector must equal number of cells");
        std::vector<double> soa(size_t(m->n_state) * m->n);
        for (int64_t i = 0; i < m->n; ++i)
            for (int s = 0; s < m->n_state; ++s) soa[size_t(s) * m->n + i] = states[i * m->n_state + s];
        m->d_initial_state.upload(soa, m->stream);
        CUDA_OK(cudaStreamSynchronize(m->stream));
        m->has_initial = true;
    });
}
int sb2_get_initial_state(const sb2_model* m, double* states, int64_t n_cells) {
    return guarded_c(m, [&] {
        if (n_cells != m->n) throw Error("Length of the state vector must equal number of cells");
        if (!m->has_initial) throw Error("Initial state not yet established or set");
        std::vector<double> soa(size_t(m->n_state) * m->n);
        CUDA_OK(cudaMemcpyAsync(soa.data(), m->d_initial_state.p, soa.size() * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
        CUDA_OK(cudaStreamSynchronize(m->stream));
        for (int64_t i = 0; i < m->n; ++i)
            for (int s = 0; s < m->n_state; ++s) states[i * m->n_state + s] = soa[size_t(s) * m->n + i];
    });
}
int sb2_revert_to_initial_state(sb2_model* m) {
    return guarded(m, [&] {
        if (!m->has_initial) throw Error("Initial state not yet established or set");
        CUDA_OK(cudaMemcpyAsync(m->d_state.p, m->d_initial_state.p, m->d_state.n * sizeof(double), cudaMemcpyDeviceToDevice, m->stream));
    });
}
int sb2_adjust_q(sb2_model* m, double q_scale, const int64_t* cids, int n) {
    return guarded(m, [&] {
        // state.adjust_q: kirchner.q *= q_scale (pt_gs_k.h:219-221, pt_hs_k.h:164); hbv_stack scales soil.sm, tank.uz, tank.lz (hbv_stack.h:182-185)
        std::vector<uint8_t> sel(m->n, n == 0 ? 1 : 0);
        for (int64_t i = 0; i < m->n && n > 0; ++i)
            for (int k = 0; k < n; ++k)
                if (m->geo[i].catchment_id == cids[k]) { sel[i] = 1; break; }
        DevArray<uint8_t> d_sel;
        d_sel.upload(sel, m->stream);
        const int first = m->stack == SB2_HBV_STACK ? m->n_state - 3 : m->n_state - 1;
        for (int s = first; s < m->n_state; ++s) {
            scale_selected_kernel<<<grid_for(m->n, 256), 256, 0, m->stream>>>(m->d_state.p + size_t(s) * m->n, d_sel.p, m->n, q_scale);
            ++m->launches;
        }
        CUDA_OK(cudaGetLastError());
        CUDA_OK(cudaStreamSynchronize(m->stream));
    });
}
// ---- cell-identified state io: state_io_handler (api/api_state.h:93-142) -------------------------------------------------
namespace {
struct StateIdLess {
    bool operator()(const sb2_cell_state_id& a, const sb2_cell_state_id& b) const {  // cell_state_id::operator< (:46-54)
        if (a.cid != b.cid) return a.cid < b.cid;
        if (a.x != b.x) return a.x < b.x;
        if (a.y != b.y) return a.y < b.y;
        return a.area < b.area;
    }
};
sb2_cell_state_id cell_state_id_of(const sb2_geo_cell& g) {  // :58-60, the coordinates and the area go through int
    return sb2_cell_state_id{g.catchment_id, int64_t(int(g.x)), int64_t(int(g.y)), int64_t(int(g.area))};
}
bool cid_in_scope(const int64_t* cids, int n, int64_t cid) { return n == 0 || std::find(cids, cids + n, cid) != cids + n; }
}  // namespace

int sb2_extract_state(const sb2_model* cm, const int64_t* cids, int n_cids, sb2_cell_state_id* ids, double* states, int64_t* n_out) {
    return guarded_c(cm, [&] {
        sb2_model* m = const_cast<sb2_model*>(cm);
        if (!n_out || (n_cids > 0 && !cids)) throw Error("null argument");
        std::vector<int64_t> cells;
        for (int64_t i = 0; i < m->n; ++i)
            if (cid_in_scope(cids, n_cids, m->geo[size_t(i)].catchment_id)) cells.push_back(i);
        *n_out = int64_t(cells.size());
        if (cells.empty()) return;
        if (!ids || !states) throw Error("null output");
        for (size_t k = 0; k < cells.size(); ++k) ids[k] = cell_state_id_of(m->geo[size_t(cells[k])]);
        DevArray<int64_t> d_cells;
        DevArray<double> d_out;
        d_cells.upload(cells, m->stream);
        const int64_t total = int64_t(cells.size()) * m->n_state;
        d_out.resize(size_t(total));
        state_gather_kernel<<<grid_for(total, 256), 256, 0, m->stream>>>(m->d_state.p, m->n, m->n_state, d_cells.p, int64_t(cells.size()), d_out.p);
        CUDA_OK(cudaGetLastError());
        ++m->launches;
        CUDA_OK(cudaMemcpyAsync(states, d_out.p, size_t(total) * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
        CUDA_OK(cudaStreamSynchronize(m->stream));
    });
}
int sb2_apply_state(sb2_model* m, int64_t n, const sb2_cell_state_id* ids, const double* states, const int64_t* cids, int n_cids, int64_t* missing,
                    int64_t* n_missing) {
    return guarded(m, [&] {
        if (n < 0 || (n > 0 && (!ids || !states)) || (n_cids > 0 && !cids) || !n_missing) throw Error("null argument");
        std::map<sb2_cell_state_id, int64_t, StateIdLess> cmap;  // cells in scope by id; a later cell with the same id replaces an earlier one
        for (int64_t i = 0; i < m->n; ++i)
            if (cid_in_scope(cids, n_cids, m->geo[size_t(i)].catchment_id)) cmap[cell_state_id_of(m->geo[size_t(i)])] = i;
        std::map<int64_t, int64_t> row_of_cell;  // the last state applied to a cell wins, as in the sequential loop
        *n_missing = 0;
        for (int64_t k = 0; k < n; ++k) {
            if (!cid_in_scope(cids, n_cids, ids[k].cid)) continue;
            auto f = cmap.find(ids[k]);
            if (f != cmap.end()) row_of_cell[f->second] = k;
            else {
                if (!missing) throw Error("null output");
                missing[(*n_missing)++] = k;
            }
        }
        if (row_of_cell.empty()) return;
        std::vector<int64_t> cells;
        std::vector<double> rows;
        for (auto& kv : row_of_cell) {
            cells.push_back(kv.first);
            rows.insert(rows.end(), states + kv.second * m->n_state, states + (kv.second + 1) * m->n_state);
        }
        DevArray<int64_t> d_cells;
        DevArray<double> d_rows;
        d_cells.upload(cells, m->stream);
        d_rows.upload(rows, m->stream);
        const int64_t total = int64_t(rows.size());
        state_scatter_kernel<<<grid_for(total, 256), 256, 0, m->stream>>>(m->d_state.p, m->n, m->n_state, d_cells.p, int64_t(cells.size()), d_rows.p);
        CUDA_OK(cudaGetLastError());
        ++m->launches;
        CUDA_OK(cudaStreamSynchronize(m->stream));
    });
}
int sb2_set_collector_mode(sb2_model* m, int collect_bits) {
    return guarded(m, [&] {
        if (collect_bits < 0 || collect_bits > 15) throw Error("collector mode out of range");
        if (collect_bits != m->collect_bits) free_series(m);
        m->collect_bits = collect_bits;
    });
}

// ---- environment -----------------------------------------------------------------------------------------------------
int sb2_initialize_cell_environment(sb2_model* m, int64_t t0_us, int64_t dt_us, int64_t n) {
    return guarded(m, [&] {
        if (dt_us <= 0 || n < 0) throw Error("initialize_cell_environment: invalid time axis");
        const bool same_dt = dt_us == m->dt;
        m->t0 = t0_us; m->dt = dt_us; m->T = n;
        if (!same_dt) { m->param_dirty = true; m->route.reset(); }  // the albedo decay steps and the unit hydrographs depend on dt
        std::vector<int2> doy_soy(n);
        m->h_prior_gradient.resize(n);
        for (int64_t i = 0; i < n; ++i) {
            const int64_t t = t0_us + i * dt_us;
            doy_soy[i] = make_int2(host::day_of_year(t), int32_t(host::seconds_of_year(t)));
            m->h_prior_gradient[i] = host::btk_prior_gradient(t, dt_us);
        }
        m->d_doy_soy.upload(doy_soy, m->stream);
        m->d_prior_gradient.upload(m->h_prior_gradient, m->stream);
        m->d_cq.resize(size_t(n) * m->n_catch());
        m->d_cc.resize(size_t(n) * m->n_catch());
        if (n) {
            CUDA_OK(cudaMemsetAsync(m->d_cq.p, 0, m->d_cq.n * sizeof(double), m->stream));
            CUDA_OK(cudaMemsetAsync(m->d_cc.p, 0, m->d_cc.n * sizeof(double), m->stream));
        }
        // cell.env_ts is re-created NaN-filled on demand (cell_model.h:58-72); drop whatever was there
        for (auto& f : m->d_forcing) f.release();
        m->forcing_rows = 0; m->forcing_first = 0;
        free_series(m);
        m->ran_steps = 0;
        // everything that was laid out on the PREVIOUS axis goes with it: the station series ([T_old][n_src] -- interpolating them over a
        // longer or shifted axis would read past their end or pair them with the wrong times), the interpolation plans and kriging
        // operators built on them, the cached point times of the axis, and the calibration targets (aligned against the old t0 / dt).
        // interpolate / run_windowed then see unset sources (forcing stays NaN, as for a variable without sources) and
        // calculate_goal_function asks for targets again.
        for (int v = 0; v < SB2_N_FORCING; ++v) {
            Source& src = m->src[v];
            src.n_src = 0;
            src.xyz.clear(); src.h_values.clear();
            src.d_xyz.release(); src.d_values.release();
            src.has_nonfinite = false;
            m->idw[v].valid = false; m->idw[v].dense_valid = false;
        }
        m->btk_cache.clear();
        m->d_axis_t.release();
        m->targets.clear();
        m->rlocal_valid = m->rnet_valid = false;
        CUDA_OK(cudaStreamSynchronize(m->stream));
    });
}

int sb2_set_cell_forcing(sb2_model* m, int var, const double* values, int layout) {
    return guarded(m, [&] {
        if (var < 0 || var >= SB2_N_FORCING) throw Error("unknown forcing variable");
        if (!(m->T > 0)) throw Error("initialize_cell_environment has not been called");
        ensure_forcing(m, 0, m->T, true);
        const size_t count = size_t(m->T) * m->n;
        if (layout == SB2_TIME_MAJOR) {
            CUDA_OK(cudaMemcpyAsync(m->d_forcing[var].p, values, count * sizeof(double), cudaMemcpyHostToDevice, m->stream));
        } else {
            DevArray<double> tmp;
            tmp.upload(values, count, m->stream);
            dim3 b(32, 8), g((unsigned)((m->T + 31) / 32), (unsigned)((m->n + 31) / 32));
            transpose_kernel<<<g, b, 0, m->stream>>>(tmp.p, m->d_forcing[var].p, m->n, m->T);
            CUDA_OK(cudaGetLastError());
            ++m->launches;
            CUDA_OK(cudaStreamSynchronize(m->stream));
        }
        CUDA_OK(cudaStreamSynchronize(m->stream));
    });
}
int sb2_get_cell_forcing(const sb2_model* cm, int var, int64_t start_step, int64_t n_steps, double* out, int layout) {
    return guarded_c(cm, [&] {
        sb2_model* m = const_cast<sb2_model*>(cm);
        if (var < 0 || var >= SB2_N_FORCING) throw Error("unknown forcing variable");
        if (!m->d_forcing[var].p) throw Error("cell environment not initialised");
        if (start_step < m->forcing_first || start_step + n_steps > m->forcing_first + m->forcing_rows)
            throw Error("requested steps are outside the resident forcing window");
        copy_out_2d(m, m->d_forcing[var].p + (start_step - m->forcing_first) * m->n, n_steps, out, layout);
    });
}

// common part of sb2_set_sources / sb2_set_sources_on_axis: returns the Source with its geometry installed, plans invalidated
static Source* begin_sources(sb2_model* m, int var, int64_t n_src, const double* xyz) {
    if (var < 0 || var >= SB2_N_FORCING) throw Error("unknown forcing variable");
    if (!(m->T > 0)) throw Error("initialize_cell_environment has not been called");
    Source& s = m->src[var];
    s.n_src = n_src;
    m->idw[var].valid = false;
    if (var == SB2_TEMPERATURE) m->btk_cache.clear();
    if (n_src == 0) { s.xyz.clear(); s.h_values.clear(); s.d_xyz.release(); s.d_values.release(); return nullptr; }
    s.xyz.assign(xyz, xyz + 3 * n_src);
    s.d_xyz.upload(s.xyz, m->stream);
    return &s;
}
int sb2_set_sources(sb2_model* m, int var, int64_t n_src, const double* xyz, const double* values) {
    return guarded(m, [&] {
        Source* sp = begin_sources(m, var, n_src, xyz);
        if (!sp) return;
        Source& s = *sp;
        const size_t count = size_t(m->T) * n_src;
        s.d_values.upload(values, count, m->stream);
        // average_accessor of a stair-case source on the model axis (time_series.h:202-310,2033-2072)
        // ... which also reports whether any value is NaN / inf: the scan of the values runs on the device, not over the host buffer
        m->d_scan_flag.ensure(1);
        CUDA_OK(cudaMemsetAsync(m->d_scan_flag.p, 0, sizeof(int), m->stream));
        average_accessor_same_axis_kernel<<<std::min<int64_t>(grid_for(count, 256), 148 * 16), 256, 0, m->stream>>>(s.d_values.p, int64_t(count),
                                                                                                             double(m->dt) / 1e6, m->d_scan_flag.p);
        CUDA_OK(cudaGetLastError());
        ++m->launches;
        int flag = 0;
        CUDA_OK(cudaMemcpyAsync(&flag, m->d_scan_flag.p, sizeof(int), cudaMemcpyDeviceToHost, m->stream));
        CUDA_OK(cudaStreamSynchronize(m->stream));
        s.has_nonfinite = flag != 0;
        // the host copy serves the valid-station bookkeeping of Bayesian kriging (run_btk), needed only when stations drop out
        if (var == SB2_TEMPERATURE && s.has_nonfinite) s.h_values.assign(values, values + count);
        else s.h_values.clear();
    });
}
int sb2_set_sources_on_axis(sb2_model* m, int var, int64_t n_src, const double* xyz, int64_t n_points, const int64_t* t_us, int64_t t_end_us,
                            const double* values, int point_interpretation) {
    return guarded(m, [&] {
        if (n_src > 0 && n_points > 0) {
            if (!t_us || !values) throw Error("set_sources_on_axis: null time or value array");
            for (int64_t i = 1; i < n_points; ++i)
                if (!(t_us[i] > t_us[i - 1])) throw Error("set_sources_on_axis: point times must be strictly increasing");
            if (t_end_us < t_us[n_points - 1]) throw Error("set_sources_on_axis: the total period ends before the last point");
        }
        Source* sp = begin_sources(m, var, n_src, xyz);
        if (!sp) return;
        Source& s = *sp;
        const size_t count = size_t(m->T) * n_src;
        DevArray<int64_t> d_t;
        DevArray<double> d_pts;
        d_t.upload(t_us, size_t(n_points), m->stream);
        d_pts.upload(values, size_t(n_points) * n_src, m->stream);
        s.d_values.resize(count);
        average_accessor_kernel<<<grid_for(int64_t(count), 256), 256, 0, m->stream>>>(d_t.p, d_pts.p, n_points, n_src, t_end_us,
                                                                                     point_interpretation == SB2_POINT_INSTANT_VALUE ? 1 : 0, m->t0, m->dt,
                                                                                     m->T, s.d_values.p);
        CUDA_OK(cudaGetLastError());
        ++m->launches;
        // the projected series back on the host: NaN bookkeeping of interpolate(), BTK validity sets
        std::vector<double> h(count);
        CUDA_OK(cudaMemcpyAsync(h.data(), s.d_values.p, count * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
        CUDA_OK(cudaStreamSynchronize(m->stream));
        s.has_nonfinite = false;
        for (size_t i = 0; i < count && !s.has_nonfinite; ++i) s.has_nonfinite = !std::isfinite(h[i]);
        if (var == SB2_TEMPERATURE) s.h_values = std::move(h);
    });
}
int sb2_set_sources_on_axes(sb2_model* m, int var, int64_t n_src, const double* xyz, const int64_t* n_points, const int64_t* t_us,
                            const int64_t* t_end_us, const double* values, const int32_t* point_interpretation) {
    return guarded(m, [&] {
        std::vector<int64_t> off(size_t(std::max<int64_t>(n_src, 0)) + 1, 0);
        if (n_src > 0) {
            if (!n_points || !t_us || !t_end_us || !values || !point_interpretation) throw Error("set_sources_on_axes: null argument");
            for (int64_t s = 0; s < n_src; ++s) {
                if (n_points[s] < 0) throw Error("set_sources_on_axes: negative point count");
                off[size_t(s) + 1] = off[size_t(s)] + n_points[s];
                const int64_t* t = t_us + off[size_t(s)];
                for (int64_t i = 1; i < n_points[s]; ++i)
                    if (!(t[i] > t[i - 1])) throw Error("set_sources_on_axes: point times must be strictly increasing");
                if (n_points[s] > 0 && t_end_us[s] < t[n_points[s] - 1]) throw Error("set_sources_on_axes: the total period ends before the last point");
            }
        }
        Source* sp = begin_sources(m, var, n_src, xyz);
        if (!sp) return;
        Source& s = *sp;
        const size_t count = size_t(m->T) * n_src, total = size_t(off.back());
        DevArray<int64_t> d_t, d_off, d_end;
        DevArray<double> d_pts;
        DevArray<int32_t> d_lin;
        std::vector<int32_t> lin(static_cast<size_t>(n_src), 0);
        for (int64_t k = 0; k < n_src; ++k) lin[size_t(k)] = point_interpretation[k] == SB2_POINT_INSTANT_VALUE ? 1 : 0;
        d_t.upload(t_us, total, m->stream);
        d_pts.upload(values, total, m->stream);
        d_off.upload(off, m->stream);
        d_end.upload(t_end_us, size_t(n_src), m->stream);
        d_lin.upload(lin, m->stream);
        s.d_values.resize(count);
        average_accessor_ragged_kernel<<<grid_for(int64_t(count), 256), 256, 0, m->stream>>>(d_t.p, d_pts.p, d_off.p, d_end.p, d_lin.p, n_src, m->t0, m->dt,
                                                                                            m->T, s.d_values.p);
        CUDA_OK(cudaGetLastError());
        ++m->launches;
        std::vector<double> h(count);  // NaN bookkeeping of interpolate(), BTK validity sets -- as sb2_set_sources_on_axis
        CUDA_OK(cudaMemcpyAsync(h.data(), s.d_values.p, count * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
        CUDA_OK(cudaStreamSynchronize(m->stream));
        s.has_nonfinite = false;
        for (size_t i = 0; i < count && !s.has_nonfinite; ++i) s.has_nonfinite = !std::isfinite(h[i]);
        if (var == SB2_TEMPERATURE) s.h_values = std::move(h);
    });
}
int sb2_get_sources_on_model_axis(const sb2_model* cm, int var, double* out) {
    return guarded_c(cm, [&] {
        sb2_model* m = const_cast<sb2_model*>(cm);
        if (var < 0 || var >= SB2_N_FORCING) throw Error("unknown forcing variable");
        const Source& s = m->src[var];
        if (s.n_src == 0 || !s.d_values.p) throw Error("no sources set for this variable");
        CUDA_OK(cudaMemcpyAsync(out, s.d_values.p, size_t(m->T) * s.n_src * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
        CUDA_OK(cudaStreamSynchronize(m->stream));
    });
}

int sb2_interpolate(sb2_model* m, const sb2_interpolation_parameter* ip, int best_effort, int* all_ok) {
    return guarded(m, [&] {
        if (all_ok) *all_ok = 0;
        if (!(m->T > 0)) throw Error("initialize_cell_environment has not been called");
        set_interpolation_parameter(m, ip);
        ensure_forcing(m, 0, m->T, true);
        time_begin(m, 0);
        const bool ok = interpolate_range(m, 0, m->T, best_effort);
        m->last_interp_ms = time_end(m, 0, 1);
        if (all_ok) *all_ok = ok ? 1 : 0;
    });
}

int sb2_is_cell_env_ts_ok(sb2_model* m, int* ok) {
    return guarded(m, [&] {
        // region_model.h:954-962: every env_ts value of every calculated cell is finite
        if (!m->d_forcing[0].p) { *ok = 0; return; }
        sync_filter(m);
        DevArray<unsigned long long> cnt;
        cnt.resize(1);
        CUDA_OK(cudaMemsetAsync(cnt.p, 0, sizeof(unsigned long long), m->stream));
        for (auto& f : m->d_forcing) {
            count_nonfinite_kernel<<<148 * 8, 256, 0, m->stream>>>(f.p, m->forcing_rows, m->n, m->d_active.p, cnt.p);
            ++m->launches;
        }
        CUDA_OK(cudaGetLastError());
        unsigned long long h = 0;
        CUDA_OK(cudaMemcpyAsync(&h, cnt.p, sizeof(h), cudaMemcpyDeviceToHost, m->stream));
        CUDA_OK(cudaStreamSynchronize(m->stream));
        *ok = h == 0 ? 1 : 0;
    });
}

namespace {
// region_model::run_cells (core/region_model.h:578-597) on the resident cell environment
void run_cells_resident(sb2_model* m, int start_step, int n_steps) {
    validate_run_args(m, start_step, n_steps);
    if (!m->d_forcing[0].p || m->forcing_first != 0 || m->forcing_rows != m->T)
        throw Error("run_cells: cell environment is not resident for the whole time axis (use interpolate / set_cell_forcing, or run_windowed)");
    snapshot_initial_state_if_unset(m);
    const int64_t first = n_steps > 0 ? start_step : 0;  // pt_gs_k.h:358-359: n_steps == 0 runs the whole axis
    const int64_t count = n_steps > 0 ? n_steps : m->T;
    const bool fresh = m->out_rows != m->T || m->out_first != 0;
    ensure_series(m, 0, m->T);
    // begin_run -> ts_init (cell_model.h:135-138,163-170): new series are NaN everywhere, existing ones NaN over the run range
    for (int r = 0; r < SB2_N_RESPONSE; ++r)
        if (m->d_resp[r].p) fill_nan(m, m->d_resp[r].p + (fresh ? 0 : first * m->n), (fresh ? m->T : count) * m->n);
    for (int s = 0; s < SB2_N_STATE_SERIES; ++s)
        if (m->d_st[s].p) fill_nan(m, m->d_st[s].p + (fresh ? 0 : first * m->n), (fresh ? m->T + 1 : count + 1) * m->n);
    time_begin(m, 2);
    launch_step_range(m, first, count, true);
    m->last_step_ms = time_end(m, 2, 3);
    m->ran_first = first; m->ran_steps = count;
    m->rlocal_valid = m->rnet_valid = false;
    check_device_errors(m);
}
}  // namespace

// ---- the hot path ----------------------------------------------------------------------------------------------------
int sb2_run_cells(sb2_model* m, int start_step, int n_steps) {
    return guarded(m, [&] { run_cells_resident(m, start_step, n_steps); });
}

// ---- state tuning (SURVEY 8f item 3) -------------------------------------------------------------------------------------
// region_model::adjust_state_to_target_flow (core/region_model.h:626-637) over adjust_state_model::{discharge, tune_flow}
// (core/model_state_tuning.h:38-118).  One evaluation of discharge(q_scale) stays on the device: state snapshot s0 copied back
// device-to-device, the ground-storage rows scaled for the selected cells, run_cells over [i0, i0 + n), the selected cells'
// avg_discharge rows reduced by stat_reduce_rows_kernel; only the n row sums come back to the host, where dlib's one-dimensional
// minimiser (restated in sb2_host.hpp) picks the next q_scale.
int sb2_adjust_state_to_target_flow(sb2_model* m, double wanted_flow_m3s, const int64_t* cids, int n_cids, int64_t start_step, double scale_range,
                                    double scale_eps, int64_t max_iter, int64_t n_steps, sb2_q_adjust_result* result) {
    return guarded(m, [&] {
        if (!result) throw Error("null result");
        result->q_0 = result->q_r = 0.0;
        result->diagnostics[0] = 0;
        auto set_diag = [&](const std::string& d) {
            std::snprintf(result->diagnostics, sizeof(result->diagnostics), "%s", d.c_str());
        };
        if (n_cids > 0 && !cids) throw Error("null catchment id list");
        const std::vector<uint8_t> old_filter = m->catchment_filter;
        // adjust_state_model ctor: filter := cids (throws for unknown ids, outside the reference's try block), s0 := get_states
        if (n_cids > 0) {
            if (int64_t(n_cids) > m->n_catch()) throw Error("set_catchment_calculation_filter: supplied list > available catchments");
            for (int i = 0; i < n_cids; ++i)
                if (!m->cid_to_cix.count(cids[i])) throw Error("set_catchment_calculation_filter: no cells have supplied cid");
            m->catchment_filter.assign(size_t(m->n_catch()), 0);
            for (int i = 0; i < n_cids; ++i) m->catchment_filter[size_t(m->cid_to_cix[cids[i]])] = 1;
        } else
            m->catchment_filter.clear();
        m->filter_dirty = true;
        std::vector<uint8_t> sel(size_t(m->n), n_cids == 0 ? 1 : 0);
        if (n_cids > 0)
            for (int64_t i = 0; i < m->n; ++i) sel[size_t(i)] = m->catchment_filter[size_t(m->cix_of_cell[i])];
        DevArray<uint8_t> d_sel;
        DevArray<double> d_s0, d_rows;
        d_sel.upload(sel, m->stream);
        d_s0.resize(m->d_state.n);
        CUDA_OK(cudaMemcpyAsync(d_s0.p, m->d_state.p, m->d_state.n * sizeof(double), cudaMemcpyDeviceToDevice, m->stream));
        const int first_q = m->stack == SB2_HBV_STACK ? m->n_state - 3 : m->n_state - 1;
        auto adjust_from_s0 = [&](double q_scale) {  // revert_to_state_0(); rm.adjust_q(q_scale, cids)
            CUDA_OK(cudaMemcpyAsync(m->d_state.p, d_s0.p, m->d_state.n * sizeof(double), cudaMemcpyDeviceToDevice, m->stream));
            for (int s = first_q; s < m->n_state; ++s) {
                scale_selected_kernel<<<grid_for(m->n, 256), 256, 0, m->stream>>>(m->d_state.p + size_t(s) * m->n, d_sel.p, m->n, q_scale);
                ++m->launches;
            }
            CUDA_OK(cudaGetLastError());
        };
        std::vector<double> rows;
        auto discharge = [&](double q_scale) -> double {  // model_state_tuning.h:59-73
            adjust_from_s0(q_scale);
            run_cells_resident(m, int(start_step), int(n_steps));
            const double* q = stat_series_rows(m, SB2_STAT_RESPONSE, SB2_R_AVG_DISCHARGE, start_step, n_steps);
            d_rows.resize(size_t(n_steps));
            rows.resize(size_t(n_steps));
            stat_reduce_rows_kernel<<<int(std::min<int64_t>(n_steps, 148 * 8)), 256, 0, m->stream>>>(q, m->n, n_steps, d_sel.p, nullptr, m->d_area.p,
                                                                                                     nullptr, d_rows.p);
            CUDA_OK(cudaGetLastError());
            ++m->launches;
            CUDA_OK(cudaMemcpyAsync(rows.data(), d_rows.p, rows.size() * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
            CUDA_OK(cudaStreamSynchronize(m->stream));
            double q_sum = 0.0;
            for (double v : rows) q_sum += v;
            return q_sum / double(n_steps);
        };
        auto restore_filter = [&] { m->catchment_filter = old_filter; m->filter_dirty = true; };
        try {  // region_model.h:630-634
            sb2_q_adjust_result r{};
            r.q_0 = discharge(1.0);
            double scale = wanted_flow_m3s / r.q_0;
            std::string diag;
            try {
                if (!std::isfinite(r.q_0)) throw Error("the initial simulated discharge is nan");
                host::find_min_single_variable(
                    [&](double x) { const double d = discharge(x) - wanted_flow_m3s; return d * d; }, scale, scale / scale_range, scale * scale_range,
                    scale * scale_eps, long(max_iter));
            } catch (const std::exception& e) {
                diag = "failed to find solution within " + std::to_string(max_iter) + ", exception was:" + e.what();
            }
            r.q_r = discharge(scale);
            adjust_from_s0(scale);
            CUDA_OK(cudaStreamSynchronize(m->stream));
            result->q_0 = r.q_0;
            result->q_r = r.q_r;
            set_diag(diag);
        } catch (const std::exception& e) {
            set_diag(std::string("Failed to tune_flow") + e.what());
        }
        restore_filter();
    });
}

int sb2_run_windowed(sb2_model* m, const sb2_interpolation_parameter* ip, int start_step, int n_steps, int window_steps) {
    return guarded(m, [&] {
        validate_run_args(m, start_step, n_steps);
        if (window_steps <= 0) throw Error("run_windowed: window_steps must be positive");
        set_interpolation_parameter(m, ip);
        snapshot_initial_state_if_unset(m);
        const int64_t first = n_steps > 0 ? start_step : 0;
        const int64_t count = n_steps > 0 ? n_steps : m->T;
        const int64_t W = std::min<int64_t>(window_steps, count);
        float interp_ms = 0.f, step_ms = 0.f;
        // routing over a windowed run: each window's cell discharge is convolved into the rivers' local inflow right away
        // (the per-cell series of earlier windows are gone afterwards); the last cell_max_len-1 rows are carried over
        const bool route = !m->rivers.empty() && (m->collect_bits & SB2_COLLECT_DISCHARGE) && first == 0 && count == m->T;
        int64_t H = 0;
        if (route) {
            ensure_routing_plan(m);
            H = m->route->cell_max_len - 1;
            m->d_qhist.resize(size_t(H + W) * m->n);
            CUDA_OK(cudaMemsetAsync(m->d_qhist.p, 0, size_t(H) * m->n * sizeof(double), m->stream));
            m->d_rlocal.resize(size_t(m->route->n_riv) * m->T);
        }
        m->rlocal_valid = m->rnet_valid = false;
        for (int64_t w0 = first; w0 < first + count; w0 += W) {
            const int64_t wn = std::min<int64_t>(W, first + count - w0);
            NvtxRange nv_window("window " + std::to_string((w0 - first) / W));
            // the window buffers are reused: forcing rows [w0, w0+W), series rows likewise
            if (m->forcing_rows != W || !m->d_forcing[0].p) {
                for (auto& f : m->d_forcing) f.resize(size_t(W) * m->n);
                m->forcing_rows = W;
            }
            m->forcing_first = w0;
            // a variable without sources reads NaN; so do the cells outside the calculation filter, which interpolation skips
            // (the reused window buffers would otherwise show them the previous window's or the previous run's values)
            const bool filtered = !m->catchment_filter.empty();
            for (int v = 0; v < SB2_N_FORCING; ++v)
                if (m->src[v].n_src == 0 || filtered) fill_nan(m, m->d_forcing[v].p, W * m->n);
            time_begin(m, 0);
            interpolate_range(m, w0, wn, 0);
            CUDA_OK(cudaEventRecord(m->ev[1], m->stream));
            ensure_series(m, w0, W);
            CUDA_OK(cudaEventRecord(m->ev[2], m->stream));
            launch_step_range(m, w0, wn, true);
            if (route) {
                NvtxRange nv_route("routing local inflow");
                double* row0 = m->d_qhist.p + size_t(H) * m->n;
                CUDA_OK(cudaMemcpyAsync(row0, m->d_resp[SB2_R_AVG_DISCHARGE].p, size_t(wn) * m->n * sizeof(double), cudaMemcpyDeviceToDevice, m->stream));
                routing_local_inflow(*m->route, row0, m->n, wn, H, w0, m->T, m->d_rlocal.p, m->stream, &m->launches);
                // the last H rows of [history ; window] become the history of the next window: rows [wn, wn + H) -> [0, H).  With wn < H
                // (window_steps below the longest unit hydrograph, or a short window) the two ranges overlap, which cudaMemcpy does not
                // allow: moved in ascending pieces of at most wn rows, each piece's source lying wholly behind its destination.
                if (H > 0 && w0 + wn < first + count) {
                    for (int64_t r = 0; r < H; r += wn) {
                        const int64_t rows = std::min<int64_t>(wn, H - r);
                        CUDA_OK(cudaMemcpyAsync(m->d_qhist.p + size_t(r) * m->n, m->d_qhist.p + size_t(r + wn) * m->n, size_t(rows) * m->n * sizeof(double),
                                                cudaMemcpyDeviceToDevice, m->stream));
                    }
                }
            }
            CUDA_OK(cudaEventRecord(m->ev[3], m->stream));
            CUDA_OK(cudaEventSynchronize(m->ev[3]));
            float a = 0.f, b = 0.f;
            CUDA_OK(cudaEventElapsedTime(&a, m->ev[0], m->ev[1]));
            CUDA_OK(cudaEventElapsedTime(&b, m->ev[2], m->ev[3]));
            interp_ms += a; step_ms += b;
        }
        m->last_interp_ms = interp_ms; m->last_step_ms = step_ms;
        m->ran_first = first; m->ran_steps = count;
        if (route) m->rlocal_valid = true;
        check_device_errors(m);
    });
}

// ---- results -----------------------------------------------------------------------------------------------------------
int sb2_get_response(const sb2_model* cm, int series, int64_t start_step, int64_t n_steps, double* out, int layout) {
    return guarded_c(cm, [&] {
        sb2_model* m = const_cast<sb2_model*>(cm);
        if (series < 0 || series >= SB2_N_RESPONSE) throw Error("unknown response series");
        if (!m->d_resp[series].p) throw Error("response series is not collected in the current collector mode");
        if (start_step < m->out_first || start_step + n_steps > m->out_first + m->out_rows)
            throw Error("requested steps are outside the resident series window");
        copy_out_2d(m, m->d_resp[series].p + (start_step - m->out_first) * m->n, n_steps, out, layout);
    });
}
int sb2_get_state_series(const sb2_model* cm, int series, int64_t start_step, int64_t n_points, double* out, int layout) {
    return guarded_c(cm, [&] {
        sb2_model* m = const_cast<sb2_model*>(cm);
        if (series < 0 || series >= SB2_N_STATE_SERIES) throw Error("unknown state series");
        if (!m->d_st[series].p) throw Error("state series is not collected in the current collector mode");
        if (start_step < m->out_first || start_step + n_points > m->out_first + m->out_rows + 1)
            throw Error("requested points are outside the resident series window");
        copy_out_2d(m, m->d_st[series].p + (start_step - m->out_first) * m->n, n_points, out, layout);
    });
}
static int catchment_copy(const sb2_model* cm, const DevArray<double>& d, int64_t start_step, int64_t n_steps, double* out) {
    return guarded_c(cm, [&] {
        sb2_model* m = const_cast<sb2_model*>(cm);
        if (start_step < 0 || start_step + n_steps > m->T) throw Error("requested steps are outside the time axis");
        CUDA_OK(cudaMemcpyAsync(out, d.p + start_step * m->n_catch(), size_t(n_steps) * m->n_catch() * sizeof(double), cudaMemcpyDeviceToHost,
                                m->stream));
        CUDA_OK(cudaStreamSynchronize(m->stream));
    });
}
int sb2_catchment_discharges(const sb2_model* m, int64_t start_step, int64_t n_steps, double* out) {
    return m ? catchment_copy(m, m->d_cq, start_step, n_steps, out) : 1;
}
int sb2_catchment_charges(const sb2_model* m, int64_t start_step, int64_t n_steps, double* out) {
    return m ? catchment_copy(m, m->d_cc, start_step, n_steps, out) : 1;
}


// ---- statistics readers ------------------------------------------------------------------------------------------------
int sb2_statistics_series(const sb2_model* cm, int kind, int series, const int64_t* indexes, int n_indexes, int scope, int op, int64_t start_step,
                          int64_t n_steps, double* out) {
    return guarded_c(cm, [&] {
        sb2_model* m = const_cast<sb2_model*>(cm);
        if (op < 0 || op > 2) throw Error("unknown statistics operation");
        const std::vector<uint8_t> sel = stat_selection(m, indexes, n_indexes, scope);
        const double* rows = stat_series_rows(m, kind, series, start_step, n_steps);
        if (n_steps == 0) return;
        DevArray<uint8_t> d_sel;
        DevArray<double> d_out, d_scale;
        d_sel.upload(sel, m->stream);
        d_out.resize(size_t(n_steps));
        const double* ae_scale = stat_ae_scale(m, kind, d_scale);
        const int grid = int(std::min<int64_t>(n_steps, 148 * 8));
        stat_reduce_rows_kernel<<<grid, 256, 0, m->stream>>>(rows, m->n, n_steps, d_sel.p, op == SB2_STAT_SUM ? nullptr : m->d_area.p, m->d_area.p,
                                                             ae_scale, d_out.p);
        CUDA_OK(cudaGetLastError());
        ++m->launches;
        CUDA_OK(cudaMemcpyAsync(out, d_out.p, size_t(n_steps) * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
        CUDA_OK(cudaStreamSynchronize(m->stream));
        if (op != SB2_STAT_SUM) {
            double sum_area = 0.0;  // in cell order, as the reference accumulates it
            for (int64_t i = 0; i < m->n; ++i)
                if (sel[size_t(i)]) sum_area += m->geo[size_t(i)].area;
            if (op == SB2_STAT_AREA_AVERAGE) {  // pts_t::scale_by(1 / sum_area), cell_model.h:266
                const double inv = 1 / sum_area;
                for (int64_t t = 0; t < n_steps; ++t) out[t] *= inv;
            } else {  // average_catchment_feature_value: r / sum_area, cell_model.h:306
                for (int64_t t = 0; t < n_steps; ++t) out[t] = out[t] / sum_area;
            }
        }
    });
}
int sb2_statistics_cells(const sb2_model* cm, int kind, int series, const int64_t* indexes, int n_indexes, int scope, int64_t step, double* out,
                         int64_t* n_out) {
    return guarded_c(cm, [&] {
        sb2_model* m = const_cast<sb2_model*>(cm);
        if (m->n == 0) throw Error("no cells to make extract from");
        const std::vector<uint8_t> sel = stat_selection(m, indexes, n_indexes, scope);
        const double* row = stat_series_rows(m, kind, series, step, 1);
        std::vector<int64_t> cells;
        for (int64_t i = 0; i < m->n; ++i)
            if (sel[size_t(i)]) cells.push_back(i);
        if (n_out) *n_out = int64_t(cells.size());
        if (cells.empty()) return;
        DevArray<int64_t> d_cells;
        DevArray<double> d_out, d_scale;
        d_cells.upload(cells, m->stream);
        d_out.resize(cells.size());
        const double* ae_scale = stat_ae_scale(m, kind, d_scale);
        stat_gather_row_kernel<<<grid_for(int64_t(cells.size()), 256), 256, 0, m->stream>>>(row, d_cells.p, int64_t(cells.size()), m->d_area.p, ae_scale,
                                                                                          d_out.p);
        CUDA_OK(cudaGetLastError());
        ++m->launches;
        CUDA_OK(cudaMemcpyAsync(out, d_out.p, cells.size() * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
        CUDA_OK(cudaStreamSynchronize(m->stream));
    });
}
// basic_cell_statistics::total_area ... elevation (api/api.h:183-288): host loops in the reference's order (index-major; only
// total_area honours the scope, the land-type sums and the elevation compare catchment ids whatever the scope says)
int sb2_statistics_geo(const sb2_model* cm, int what, const int64_t* indexes, int n_indexes, int scope, double* out) {
    return guarded_c(cm, [&] {
        const sb2_model* m = cm;
        if (!out) throw Error("null output");
        if (what < 0 || what > 7) throw Error("unknown geo statistic");
        auto term = [&](const sb2_geo_cell& c) {
            switch (what) {
                case 0: return c.area;
                case 1: return c.area * c.forest;
                case 2: return c.area * c.glacier;
                case 3: return c.area * c.lake;
                case 4: return c.area * c.reservoir;
                case 5: return c.area * (1.0 - c.glacier - c.lake - c.reservoir - c.forest);
                case 6: return c.area * (1.0 - c.lake - c.reservoir);
                default: return c.z * c.area;
            }
        };
        double sum = 0.0, area_sum = 0.0;
        if (n_indexes == 0) {
            for (const auto& c : m->geo) { sum += term(c); area_sum += c.area; }
        } else {
            (void)stat_selection(m, indexes, n_indexes, scope);  // verify_cids_exist
            for (int k = 0; k < n_indexes; ++k)
                for (int64_t j = 0; j < m->n; ++j) {
                    const auto& c = m->geo[size_t(j)];
                    const bool match = what == 0 ? ((scope == SB2_SCOPE_CELL_IX && indexes[k] == j) || (scope == SB2_SCOPE_CATCHMENT_IX && c.catchment_id == indexes[k]))
                                                 : (int(c.catchment_id) == indexes[k]);
                    if (match) { sum += term(c); area_sum += c.area; }
                }
        }
        *out = what == 7 ? sum / area_sum : sum;
    });
}
// ---- routing (core/routing.h:326-383; region_model.h:909-949) ------------------------------------------------------------
int sb2_set_river_network(sb2_model* m, int64_t n_rivers, const double* rivers) {
    return guarded(m, [&] {
        std::map<int64_t, int64_t> down;
        for (int64_t i = 0; i < n_rivers; ++i) {
            const int64_t id = int64_t(rivers[6 * i]);
            if (id <= 0) throw Error("river id must be > 0");
            if (down.count(id)) throw Error("river id already exists in the network");
            down[id] = int64_t(rivers[6 * i + 1]);
        }
        for (auto& kv : down) {  // downstream must exist (or be 0) and the network must be acyclic (routing.h:215-250)
            int64_t cur = kv.second;
            size_t hops = 0;
            while (cur > 0) {
                auto f = down.find(cur);
                if (f == down.end()) throw Error("river network: downstream river id not found");
                cur = f->second;
                if (++hops > down.size()) throw Error("river network: cycle detected");
            }
        }
        m->rivers.assign(rivers, rivers + 6 * n_rivers);
        m->route.reset();
        m->rlocal_valid = m->rnet_valid = false;
    });
}

int sb2_river_flows(sb2_model* m, int64_t rid, int64_t start_step, int64_t n_steps, double* local_inflow, double* upstream_inflow,
                    double* output) {
    return guarded(m, [&] {
        if (start_step < 0 || start_step + n_steps > m->T) throw Error("requested steps are outside the time axis");
        ensure_routing_plan(m);
        auto f = m->route->ix_of_rid.find(rid);
        if (f == m->route->ix_of_rid.end()) throw Error("river network: river id " + std::to_string(rid) + " not found");
        if (!m->rlocal_valid) {  // resident run: the whole avg_discharge series is in HBM
            if (!m->d_resp[SB2_R_AVG_DISCHARGE].p || m->out_first != 0 || m->out_rows != m->T)
                throw Error("river flows need avg_discharge over the whole time axis (run_cells with a discharge collector, or run_windowed with the river network set)");
            m->d_rlocal.resize(size_t(m->route->n_riv) * m->T);
            routing_local_inflow(*m->route, m->d_resp[SB2_R_AVG_DISCHARGE].p, m->n, m->T, 0, 0, m->T, m->d_rlocal.p, m->stream, &m->launches);
            m->rlocal_valid = true;
            m->rnet_valid = false;
        }
        if (!m->rnet_valid) {
            m->d_rup.resize(size_t(m->route->n_riv) * m->T);
            m->d_rout.resize(size_t(m->route->n_riv) * m->T);
            routing_network(*m->route, m->T, m->d_rlocal.p, m->d_rup.p, m->d_rout.p, m->stream, &m->launches);
            m->rnet_valid = true;
        }
        const size_t off = size_t(f->second) * m->T + start_step, bytes = size_t(n_steps) * sizeof(double);
        if (local_inflow) CUDA_OK(cudaMemcpyAsync(local_inflow, m->d_rlocal.p + off, bytes, cudaMemcpyDeviceToHost, m->stream));
        if (upstream_inflow) CUDA_OK(cudaMemcpyAsync(upstream_inflow, m->d_rup.p + off, bytes, cudaMemcpyDeviceToHost, m->stream));
        if (output) CUDA_OK(cudaMemcpyAsync(output, m->d_rout.p + off, bytes, cudaMemcpyDeviceToHost, m->stream));
        CUDA_OK(cudaStreamSynchronize(m->stream));
    });
}

// ---- calibration (core/model_calibration.h) --------------------------------------------------------------------------------
int sb2_set_targets(sb2_model* m, int n_targets, const sb2_target* targets) {
    return guarded(m, [&] {
        if (!(m->T > 0)) throw Error("initialize_cell_environment has not been called");
        std::vector<std::unique_ptr<sb2_model::Target>> out;
        std::vector<int64_t> filter;
        bool need_snow = false;
        for (int k = 0; k < n_targets; ++k) {
            const sb2_target& s = targets[k];
            auto t = std::make_unique<sb2_model::Target>();
            if (s.n <= 0 || !s.values) throw Error("target_specification: empty target time-series");
            if (s.calc_mode < 0 || s.calc_mode > 3 || s.property < 0 || s.property > 4) throw Error("target_specification: unknown calc_mode or property");
            if (s.period_points_us) {  // point axis
                t->points.assign(s.period_points_us, s.period_points_us + s.n + 1);
                for (int64_t i = 1; i <= s.n; ++i)
                    if (!(t->points[size_t(i)] > t->points[size_t(i) - 1])) throw Error("target_specification: the axis points must be strictly increasing");
                t->d_points.upload(t->points, m->stream);
            } else if (s.dt_us <= 0) throw Error("target_specification: the target time-axis needs a positive delta_t");
            // whole runs of model steps inside the model axis are reduced in the goal kernel itself; any other fixed_dt axis goes
            // through the general projection (average_accessor_kernel), as average_accessor<pts_t, ta_t> does it (:859)
            t->aligned = !(s.period_points_us != nullptr || s.dt_us % m->dt != 0 || (s.t0_us - m->t0) % m->dt != 0 || s.t0_us < m->t0 ||
                           (s.t0_us - m->t0) / m->dt + int64_t(s.n) * (s.dt_us / m->dt) > m->T);
            t->obs.assign(s.values, s.values + s.n);
            t->t0 = s.t0_us; t->dt = s.dt_us;
            t->cids.assign(s.catchment_ids, s.catchment_ids + s.n_catchments);
            t->river_id = s.river_id; t->scale_factor = s.scale_factor; t->calc_mode = s.calc_mode; t->property = s.property;
            t->s_r = s.s_r; t->s_a = s.s_a; t->s_b = s.s_b;
            std::vector<int32_t> cix;
            if (s.property == SB2_TARGET_ROUTED_DISCHARGE) {
                cix.push_back(0);
                // catchments feeding the river (and its upstreams) are calculated (model_calibration.h:536-539)
                for (int64_t i = 0; i < m->n; ++i)
                    if (m->geo[i].routing_id > 0) filter.push_back(m->geo[i].catchment_id);
            } else {
                if (s.n_catchments <= 0) throw Error("target_specification: no catchment ids");
                for (auto cid : t->cids) {
                    auto f = m->cid_to_cix.find(cid);
                    if (f == m->cid_to_cix.end()) throw Error("target_specification: catchment id " + std::to_string(cid) + " not found");
                    if (m->catch_param.count(cid)) throw Error("Cannot calibrate on local parameters.");
                    cix.push_back(int32_t(f->second));
                    filter.push_back(cid);
                }
                if (s.property == SB2_TARGET_SNOW_COVERED_AREA || s.property == SB2_TARGET_SNOW_WATER_EQUIVALENT) {
                    need_snow = true;
                    cix.assign(1, 0);
                }
            }
            t->d_obs.upload(t->obs, m->stream);
            t->d_cix.upload(cix, m->stream);
            out.push_back(std::move(t));
        }
        CUDA_OK(cudaStreamSynchronize(m->stream));
        m->targets = std::move(out);
        // prepare_optimize (:517-552): snow collection on when a target asks for it, calculation filter = union of target catchments
        if (need_snow && !(m->collect_bits & SB2_COLLECT_SNOW)) { free_series(m); m->collect_bits |= SB2_COLLECT_SNOW; }
        std::sort(filter.begin(), filter.end());
        filter.erase(std::unique(filter.begin(), filter.end()), filter.end());
        if (!filter.empty()) {
            m->catchment_filter.assign(m->n_catch(), 0);
            for (auto cid : filter) m->catchment_filter[m->cid_to_cix[cid]] = 1;
            m->filter_dirty = true;
        }
        snapshot_initial_state_if_unset(m);
    });
}

int sb2_calculate_goal_function(sb2_model* m, const double* p, int n, double* goal) {
    if (m && sb2_set_region_parameter(m, p, n) != 0) return 1;
    if (m && sb2_revert_to_initial_state(m) != 0) return 1;
    if (m && sb2_run_cells(m, 0, 0) != 0) return 1;
    return guarded(m, [&] {
        if (m->targets.empty()) throw Error("no target specification set");
        *goal = evaluate_goal_single(m);
    });
}

int sb2_calculate_goal_function_batch(sb2_model* m, int64_t n_sets, const double* P, double* goals) {
    return guarded(m, [&] {
        if (m->targets.empty()) throw Error("no target specification set");
        if (n_sets <= 0) return;
        // pt_ss_k is not among them: its batch goes one set at a time
        bool device_batch = m->stack == SB2_PT_GS_K || m->stack == SB2_PT_HS_K || m->stack == SB2_HBV_STACK || m->stack == SB2_PT_HPS_K;
        for (auto& t : m->targets)
            if ((t->property != SB2_TARGET_DISCHARGE && t->property != SB2_TARGET_CELL_CHARGE && t->property != SB2_TARGET_ROUTED_DISCHARGE) ||
                !t->aligned)
                device_batch = false;
        if (device_batch) {
            if (!m->has_initial) throw Error("Initial state not yet established or set");
            if (!m->d_forcing[0].p || m->forcing_first != 0 || m->forcing_rows != m->T)
                throw Error("run_cells: cell environment is not resident for the whole time axis (use interpolate / set_cell_forcing, or run_windowed)");
            goal_batch(m, n_sets, P, goals);
        } else {  // one member at a time through the single-evaluation entry
            for (int64_t e = 0; e < n_sets; ++e)
                if (sb2_calculate_goal_function(m, P + e * m->n_param, m->n_param, goals + e) != 0) throw Error(m->err);
        }
    });
}

// ---- diagnostics ---------------------------------------------------------------------------------------------------------------
int sb2_unit_eval(int device, int fn, int64_t n, const double* in, int n_in, double* out, int n_out) {
    try {
        static const int need_in[UNIT_N] = {1, 1, 2, 1, 2, 5, 7, 7, 1, 1, 2, 7, 2, 7, 18, 4, 41}, need_out[UNIT_N] = {1, 1, 1, 1, 1, 1, 2, 3, 1, 1, 1, 3, 2, 3, 11, 2, 27};
        if (fn < 0 || fn >= UNIT_N) throw Error("unknown unit function");
        if (n_in < need_in[fn] || n_out < need_out[fn]) throw Error("unit function: too few input or output columns");
        CUDA_OK(cudaSetDevice(device));
        DevArray<double> d_in, d_out;
        d_in.upload(in, size_t(n) * n_in, 0);
        d_out.resize(size_t(n) * n_out);
        CUDA_OK(cudaMemsetAsync(d_out.p, 0, size_t(n) * n_out * sizeof(double), 0));
        double dtb[26];
        fill_dopri_products(1.0, dtb);
        CUDA_OK(cudaMemcpyToSymbol(kUnitDtb, dtb, sizeof(dtb)));
        unit_eval_kernel<<<grid_for(n, 128), 128, SB2_MTAB_BYTES>>>(fn, n, d_in.p, n_in, d_out.p, n_out);
        CUDA_OK(cudaGetLastError());
        CUDA_OK(cudaMemcpy(out, d_out.p, size_t(n) * n_out * sizeof(double), cudaMemcpyDeviceToHost));
        return 0;
    } catch (const std::exception& e) {
        g_create_error = e.what();
        return 1;
    }
}

int sb2_host_eval(int fn, const double* in, int n_in, double* out, int n_out) {
    try {
        if (!in || !out) return 1;
        if (fn == 0) {
            if (n_in < 8 || n_out < 4) return 1;
            const double a = in[0], b = in[1], c = in[2];
            long evals = 0;
            auto f = [&](double x) { ++evals; return (x - a) * (x - a) + b * std::cosh(x - c); };
            double x = in[3];
            out[3] = 0.0;
            try {
                out[1] = host::find_min_single_variable(f, x, in[4], in[5], in[6], long(in[7]));
            } catch (const host::MinimiserFailure&) {
                out[1] = std::nan("");
                out[3] = 1.0;
            }
            out[0] = x;
            out[2] = double(evals);
            return 0;
        }
        if (fn == 1) {
            if (n_in < 1 || n_out < 2) return 1;
            out[0] = double(host::day_of_year(int64_t(in[0])));
            out[1] = double(host::seconds_of_year(int64_t(in[0])));
            return 0;
        }
        if (fn == 2) {
            if (n_in < 3 || n_out < 1) return 1;
            const std::vector<double> w = host::make_uhg_from_gamma(int(in[0]), in[1], in[2]);
            if (int(w.size()) + 1 > n_out) return 1;
            out[0] = double(w.size());
            std::copy(w.begin(), w.end(), out + 1);
            return 0;
        }
        if (fn == 3) {
            if (n_in < 3 || n_out < 1) return 1;
            out[0] = double(host::uhg_steps(in[0], in[1], int64_t(in[2])));
            return 0;
        }
        return 1;
    } catch (const std::exception&) {
        return 1;
    }
}
int sb2_set_idw_dense(sb2_model* m, int on) {
    return guarded(m, [&] { m->force_sparse_idw = on == 0; });
}

// ---- device-side hooks -----------------------------------------------------------------------------------------------------
int sb2_set_stream(sb2_model* m, void* cuda_stream) {
    return guarded(m, [&] {
        CUDA_OK(cudaStreamSynchronize(m->stream));
        m->stream = (cudaStream_t)cuda_stream;
    });
}
int sb2_device_catchment_discharges(sb2_model* m, void** dptr, int64_t* n_steps, int64_t* n_catchments) {
    return guarded(m, [&] { *dptr = m->d_cq.p; *n_steps = m->T; *n_catchments = m->n_catch(); });
}
int sb2_device_catchment_charges(sb2_model* m, void** dptr, int64_t* n_steps, int64_t* n_catchments) {
    return guarded(m, [&] { *dptr = m->d_cc.p; *n_steps = m->T; *n_catchments = m->n_catch(); });
}
int64_t sb2_check_guards(char* message, int message_size) {
    const int64_t v = GuardZones::get().check_all();
    if (message && message_size > 0) {
        std::lock_guard<std::mutex> g(GuardZones::get().mu);
        std::snprintf(message, size_t(message_size), "%s", GuardZones::get().first.c_str());
    }
    return v;
}
int64_t sb2_kernel_launches(const sb2_model* m) { return m ? m->launches : -1; }
int sb2_step_chunk_steps(const sb2_model* m) { return m ? m->partial_steps : -1; }
int sb2_last_run_kernel_ms(const sb2_model* m, float* step_ms, float* interp_ms) {
    return guarded_c(m, [&] {
        if (step_ms) *step_ms = m->last_step_ms;
        if (interp_ms) *interp_ms = m->last_interp_ms;
    });
}

}  // extern "C"

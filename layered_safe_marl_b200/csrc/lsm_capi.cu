// lsm_capi.cu - the extern "C" boundary declared in include/lsm_b200.h.
// Host-only logic: validation, shared-memory layout, lookup tables, launch geometry.
#include <algorithm>
#include <atomic>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <functional>
#include <emmintrin.h>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "lsm_host.h"

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) { g_err = msg; return code; }
int cuda_fail(cudaError_t e, const char* what) {
    g_err = std::string(what) + ": " + cudaGetErrorString(e);
    return 100 + (int)e;
}

int next_pow2(int v) { int p = 1; while (p < v) p <<= 1; return p; }
int align_up(int v, int a) { return (v + a - 1) / a * a; }

// every entry point that touches the device runs on the handle's device and restores the caller's current device
struct DeviceGuard {
    int prev = -1; bool switched = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) switched = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
};

// ---------------------------------------------------------------------------------------------------------------
// host-side worker pool of lsm_expand_adjacency_host: persistent threads, one job (a function over [0, parts)) at a time
// ---------------------------------------------------------------------------------------------------------------
class HostPool {
public:
    static HostPool& get() { static HostPool p; return p; }
    template <class F> void run(int parts, F&& fn) {
        std::unique_lock<std::mutex> api(api_mu_);                 // one job at a time
        while ((int)threads_.size() < parts - 1) threads_.emplace_back([this] { loop(); });
        {
            std::lock_guard<std::mutex> lk(mu_);
            job_ = [&fn](int part) { fn(part); };
            parts_ = parts; next_ = 1; pending_ = parts - 1;
        }
        cv_.notify_all();
        fn(0);                                                     // the caller takes part 0
        std::unique_lock<std::mutex> lk(mu_);
        done_cv_.wait(lk, [this] { return pending_ == 0; });
        parts_ = 0; next_ = 0; job_ = nullptr;
    }
private:
    HostPool() = default;
    ~HostPool() {
        { std::lock_guard<std::mutex> lk(mu_); stop_ = true; }
        cv_.notify_all();
        for (auto& t : threads_) t.join();
    }
    void loop() {
        for (;;) {
            int part;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [this] { return stop_ || next_ < parts_; });
                if (stop_) return;
                part = next_++;
            }
            job_(part);
            {
                std::lock_guard<std::mutex> lk(mu_);
                if (--pending_ == 0) done_cv_.notify_all();
            }
        }
    }
    std::mutex api_mu_, mu_;
    std::condition_variable cv_, done_cv_;
    std::vector<std::thread> threads_;
    std::function<void(int)> job_;
    int parts_ = 0, next_ = 0, pending_ = 0;
    bool stop_ = false;
};

}  // namespace

struct lsm_handle {
    lsm::KParams kp;
    bool have_buffers = false;
    int device = 0;
    int sm_count = 0;
    int grid_cap = 0;           // sm_count * blocks_per_sm
    int warps_per_block = 0;
    int block_threads = 0;
    int smem_per_block = 0;
    int regs = 0;
    int blocks_per_sm = 0;
    uint16_t* d_pair_tab = nullptr;
    uint32_t* d_sel_tab = nullptr;
    uint32_t* d_pair32 = nullptr;
    bool spec = false;          // compile-time specialised pipeline available for (dynamics, N, L)
    int bytes_per_env = 0;      // shared memory of one environment (agent kernel: emit record + scratch)
    int epw_max = 1;            // 32 / G
    int smem_optin = 0;
    lsm::SpecTable tab = {};    // kernels and launch geometry of the specialised pipeline (spec)
    bool pairval_valid = false;         // d_pairval holds the HJ pair values of the CURRENT state (written by the last emit launch)
    double* d_pairval = nullptr;        // library-owned scratch of the specialised pipeline
    unsigned char* d_emit_rec = nullptr;
    unsigned long long* d_timeline = nullptr;   // diagnostics only (lsm_debug_timeline)
    float* d_vpacked = nullptr;          // corner-packed copy of the value grid (GridDev::packed)
    // chunked launches: big batches are split into `chunks` env ranges on library-owned streams so that the latency-bound
    // agent kernel of one range runs beside the HBM-bound emit kernel of another (fork / join with events, no host sync)
    int chunks = 1;
    std::vector<cudaStream_t> streams;
    std::vector<cudaEvent_t> ev_join;
    cudaEvent_t ev_fork = nullptr;
    float* d_grads8 = nullptr;           // padded 5-D gradient rows (GridDev::grads8)
    // fused COO edge output (lsm_set_edge_output): library-owned scratch + per-range "counts done" events
    int* d_edge_local = nullptr;
    long long* d_edge_totals = nullptr;
    long long* d_edge_block = nullptr;      // [2][edge_block_cap]: totals, then bases
    size_t edge_block_cap = 0;
    unsigned* d_edge_tickets = nullptr;
    std::vector<cudaEvent_t> ev_count;
    // host-facing step (lsm_fetch_host / lsm_step_host): range events, action staging
    std::vector<cudaEvent_t> ev_host;
    void* d_act = nullptr; void* h_act = nullptr; size_t act_bytes = 0;
    // CUDA-graph replay of the step's launches (lsm_tuning.use_graph): one graph launch instead of 2-3 kernel launches once
    // the same parameter block is seen twice in a row (fixed action / output buffers - the host-facing step, a policy
    // loop with static tensors); any change (re-pointed outputs, new episode number) takes the plain launches once and
    // re-captures on the next repeat. Captured on a library stream: the caller's stream may be the legacy default stream.
    struct GraphKey { lsm::KParams kp; int was_valid; int placement; };
    cudaStream_t g_stream = nullptr;
    cudaGraphExec_t g_exec = nullptr;
    GraphKey* g_key = nullptr;          // parameters g_exec was captured with
    GraphKey* g_seen = nullptr;         // parameters of the previous plain launch
    bool g_key_valid = false, g_seen_valid = false;
    long long g_replays = 0, g_captures = 0;
    lsm_tuning tuning = { 0, -1, -1, -1 };   // lsm_set_tuning (0 / -1 = automatic)
    int pair_placement = 0;             // 0 late (lsm_pair_kernel behind the emit kernel), 2 in front of the agent kernel, 3 between agent and emit kernel, 4 tail of the agent kernel
};

extern "C" {

int lsm_abi_version(void) { return LSM_ABI_VERSION; }
const char* lsm_last_error(void) { return g_err.c_str(); }

int lsm_create(const lsm_config* cfg, lsm_handle** out) {
    if (cfg == nullptr || out == nullptr) return fail(1, "lsm_create: null argument");
    *out = nullptr;
    const int N = cfg->num_agents, L = cfg->num_landmarks;
    if (cfg->dynamics != LSM_DYN_DOUBLE_INTEGRATOR && cfg->dynamics != LSM_DYN_AIRTAXI)
        return fail(2, "lsm_create: dynamics must be 0 (double_integrator) or 1 (airtaxi)");
    if (N < 1 || N > LSM_MAX_AGENTS) return fail(2, "lsm_create: num_agents must be in [1, 32]");
    if (L < 2) return fail(2, "lsm_create: num_landmarks (per agent) must be >= 2 (reference asserts len(goal_position) > 1)");
    if (N * L > LSM_MAX_LANDMARKS) return fail(2, "lsm_create: num_agents*num_landmarks must be <= 128 (np.int8 landmark index, Q8)");
    if (!(cfg->flags & LSM_FLAG_USE_MASKING)) return fail(2, "lsm_create: use_masking=False is not supported (reference raises, Q9)");
    if (cfg->num_internal_step < 1) return fail(2, "lsm_create: num_internal_step must be >= 1");
    if (cfg->num_total_episode < 1) return fail(2, "lsm_create: num_total_episode must be >= 1");
    if (cfg->episode_length < 1) return fail(2, "lsm_create: episode_length must be >= 1");
    if (cfg->num_obstacles < 0 || cfg->num_obstacles > LSM_MAX_OBSTACLES) return fail(2, "lsm_create: num_obstacles must be in [0, 32]");

    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(3, "lsm_create: no CUDA device - this library has no CPU fallback");
    lsm_handle* h = new lsm_handle();
    std::memset(&h->kp, 0, sizeof(h->kp));
    e = cudaGetDevice(&h->device);
    if (e != cudaSuccess) { delete h; return cuda_fail(e, "cudaGetDevice"); }
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, h->device);
    if (e != cudaSuccess) { delete h; return cuda_fail(e, "cudaGetDeviceProperties"); }
    h->sm_count = prop.multiProcessorCount;

    lsm::KParams& kp = h->kp;
    kp.c = *cfg;
    const int O = cfg->num_obstacles;           // declared extension (lsm_b200.h): entities are agents, landmarks, obstacles
    const int M = N * L, E = N + M + O;
    kp.N = N; kp.L = L; kp.M = M; kp.E = E; kp.O = O;
    kp.D = cfg->dynamics == LSM_DYN_DOUBLE_INTEGRATOR ? 7 : 6;
    kp.F = (cfg->flags & LSM_FLAG_GRAPH_FEAT_GLOBAL) ? 7 : (cfg->dynamics == LSM_DYN_DOUBLE_INTEGRATOR ? 10 : 11);
    kp.G = next_pow2(N);
    kp.EPW = 32 / kp.G;
    h->epw_max = kp.EPW;
    kp.W = (E + 31) / 32;
    kp.adj_vec = (E % 4 == 0) ? 4 : 1;
    for (int k = 0; k < 5; ++k) {
        const double stair = (double)k / 4.0;
        const double phase = stair * 0.5 * lsm::kPi;
        kp.sep_ratio_tab[k] = 1.0 - lsm_cos(phase);
    }
    // exact squared thresholds: sqrt_rn is monotone, so {t : sqrt_rn(t) >= T} is [lt(T), inf)
    {
        auto lt = [](double T) {
            if (!(T > 0.0)) return 0.0;
            double t = T * T;
            while (t > 0.0 && std::sqrt(t) >= T) t = std::nextafter(t, 0.0);
            while (std::sqrt(t) < T) t = std::nextafter(t, INFINITY);
            return t;
        };
        auto gt = [](double T) {
            if (T < 0.0) return 0.0;
            double t = T * T;
            while (t > 0.0 && std::sqrt(t) > T) t = std::nextafter(t, 0.0);
            while (!(std::sqrt(t) > T)) t = std::nextafter(t, INFINITY);
            return t;
        };
        const double R = cfg->coordination_range;
        kp.r2_lt = lt(R); kp.r2_gt = gt(R);
        // the reference's float32 adjacency drops an entity pair whose distance rounds to 0 in float32 (d <= 2^-150)
        {
            double t = std::ldexp(1.0, -300);
            while ((float)std::sqrt(t) != 0.0f) t = std::nextafter(t, 0.0);
            while ((float)std::sqrt(std::nextafter(t, INFINITY)) == 0.0f) t = std::nextafter(t, INFINITY);
            kp.r2_nz = t;
        }
        kp.col2_lt = lt(1.05 * (0.050 + 0.050));
        kp.engref2_lt = lt(cfg->engagement_distance_ref);
        kp.septgt2_lt = lt(cfg->separation_distance_target);
        for (int k = 0; k < 5; ++k) {
            // scenario.separation_distance / engagement_distance at stair level k (same expressions as the kernel)
            const double sep_ratio = kp.sep_ratio_tab[k];
            const double sep_init = (cfg->flags & LSM_FLAG_SEPARATION_DISTANCE_CURRICULUM) ? 0.0 : cfg->separation_distance_target;
            volatile double a = sep_init * (1.0 - sep_ratio);
            volatile double b = cfg->separation_distance_target * sep_ratio;
            const double sep = a + b;
            volatile double dlt = sep - cfg->engagement_ref_separation;
            const double eng = cfg->engagement_distance_ref + dlt;
            kp.sep2_lt[k] = lt(sep); kp.eng2_lt[k] = lt(eng);
        }
    }
    // shared-memory layout of one environment (generic kernel; the specialised kernels use a struct)
    lsm::SmemLayout& sl = kp.sl;
    int off = 0;
    auto take = [&](int bytes, int align) { off = align_up(off, align); int o = off; off += bytes; return o; };
    const int dN = 8 * N, dM = 8 * M, iN = 4 * N;
    sl.ax = take(dN, 8); sl.ay = take(dN, 8); sl.as2 = take(dN, 8); sl.as3 = take(dN, 8);
    sl.vpre_x = take(dN, 8); sl.vpre_y = take(dN, 8); sl.vpost_x = take(dN, 8); sl.vpost_y = take(dN, 8);
    sl.spd_post = take(dN, 8); sl.sth = take(dN, 8); sl.cth = take(dN, 8);
    sl.rawx = take(dN, 8); sl.rawy = take(dN, 8);
    sl.lx = take(dM, 8); sl.ly = take(dM, 8); sl.lh = take(dM, 8); sl.lsp = take(dM, 8);
    sl.lsin = take(dM, 8); sl.lcos = take(dM, 8);
    sl.ox = take(8 * O, 8); sl.oy = take(8 * O, 8);
    sl.daa = take(8 * N * N, 8);
    sl.dthr = take(4 * E * E, 16);
    sl.goal_pre = take(iN, 4); sl.goal_post = take(iN, 4); sl.reached_pre = take(iN, 4); sl.reached_post = take(iN, 4);
    sl.done_pre = take(iN, 4); sl.done_post = take(iN, 4);
    sl.disc_pre = take(4 * kp.W, 4); sl.disc_post = take(4 * kp.W, 4);
    sl.keepm = take(4 * N * kp.W, 4);
    sl.bytes_per_env = align_up(off, 16);
    h->smem_optin = (int)prop.sharedMemPerBlockOptin;

    // both node-feature types ('relative', which every shipped script uses, and 'global') and both interpolation
    // arithmetics run the specialised pipeline; LSM_FLAG_INTERP_FLOAT32 selects agent / pair kernels compiled with float32
    // grid lookups, so that the float64 kernels carry none of its code
    // (the obstacle extension is specialised for the shapes LSM_SPEC_LIST names with O > 0; other obstacle counts: generic)
    const bool f32 = (cfg->flags & LSM_FLAG_INTERP_FLOAT32) != 0;
    h->spec = lsm::spec_table(cfg->dynamics, N, L, O, f32, &h->tab);
    // where the next step's HJ pair values are computed (measured, DESIGN.md 3): in lsm_pair_kernel behind the emit kernel
    // ("late") for the 4-D double-integrator grid; between the agent and the emit kernel ("middle") for the 5-D airtaxi
    // grid, whose lookups are half an emit kernel's worth of work and hurt it more when they share the SMs.
    // lsm_set_tuning overrides.
    h->pair_placement = cfg->dynamics == LSM_DYN_AIRTAXI ? 3 : 0;
    if (h->spec) {
        h->bytes_per_env = h->tab.rec_bytes + h->tab.scratch_bytes;
        // agent kernel: one lane per agent, 32/N envs per warp
        h->epw_max = 32 / N; kp.EPW = h->epw_max;
        int wpb = h->tab.agent_block / 32;
        while (wpb > 1 && h->bytes_per_env * kp.EPW * wpb > h->smem_optin) --wpb;
        h->warps_per_block = wpb;
        h->block_threads = 32 * wpb;
    } else {
        h->bytes_per_env = sl.bytes_per_env;
        // as many warps per block as fit ~100 KB so that two blocks share an SM
        kp.smem_per_warp = sl.bytes_per_env * kp.EPW;
        int wpb = (100 * 1024) / kp.smem_per_warp;
        if (wpb > 8) wpb = 8;
        if (wpb < 1) wpb = 1;
        h->warps_per_block = wpb;
        h->block_threads = 32 * wpb;
    }
    kp.smem_per_warp = h->bytes_per_env * kp.EPW;
    h->smem_per_block = kp.smem_per_warp * h->warps_per_block;
    if (h->smem_per_block > h->smem_optin) {
        delete h;
        return fail(4, "lsm_create: one environment group does not fit in shared memory");
    }
    e = lsm::kernel_prepare(h->spec ? h->tab.agent : lsm::generic_ptr(cfg->dynamics), h->block_threads, h->smem_per_block, &h->regs,
                            &h->blocks_per_sm);
    if (e != cudaSuccess) { delete h; return cuda_fail(e, "kernel_prepare"); }
    if (h->blocks_per_sm < 1) { delete h; return fail(4, "lsm_create: kernel does not fit on an SM"); }
    h->grid_cap = h->sm_count * h->blocks_per_sm;
    if (h->spec) {
        if (h->tab.emit_smem > h->smem_optin) { delete h; return fail(4, "lsm_create: emit record does not fit in shared memory"); }
        e = lsm::spec_prepare(&h->tab);
        if (e != cudaSuccess) { delete h; return cuda_fail(e, "spec_prepare"); }
        if (h->tab.emit_blocks_per_sm < 1) { delete h; return fail(4, "lsm_create: emit kernel does not fit on an SM"); }
    }

    // lookup tables
    std::vector<uint16_t> pairs;
    pairs.reserve((size_t)E * (E - 1));
    for (int a = 0; a < E; ++a) for (int b = a + 1; b < E; ++b) {
        pairs.push_back((uint16_t)a); pairs.push_back((uint16_t)b);
    }
    kp.num_pairs = (int)(pairs.size() / 2);
    std::vector<uint32_t> sel((size_t)N * kp.W, 0u);
    for (int i = 0; i < N; ++i) for (int ent = 0; ent < E; ++ent) {
        if (ent >= N + M) continue;                 // obstacles have no owner (their pre / post view is the same: never disconnected)
        const int owner = ent < N ? ent : (ent - N) % N;
        if (owner <= i) sel[(size_t)i * kp.W + (ent >> 5)] |= 1u << (ent & 31);
    }
    e = cudaMalloc(&h->d_pair_tab, pairs.size() * sizeof(uint16_t));
    if (e == cudaSuccess) e = cudaMemcpy(h->d_pair_tab, pairs.data(), pairs.size() * sizeof(uint16_t), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc(&h->d_sel_tab, sel.size() * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMemcpy(h->d_sel_tab, sel.data(), sel.size() * sizeof(uint32_t), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { lsm_destroy(h); return cuda_fail(e, "table upload"); }
    std::vector<uint32_t> pair32(pairs.size() / 2);
    for (size_t k2 = 0; k2 < pair32.size(); ++k2) pair32[k2] = ((uint32_t)pairs[2 * k2] << 16) | (uint32_t)pairs[2 * k2 + 1];
    if (e == cudaSuccess) e = cudaMalloc(&h->d_pair32, pair32.size() * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMemcpy(h->d_pair32, pair32.data(), pair32.size() * sizeof(uint32_t), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { lsm_destroy(h); return cuda_fail(e, "table upload"); }
    kp.pair_tab = h->d_pair_tab; kp.sel_tab = h->d_sel_tab; kp.pair32 = h->d_pair32;
    // cos/sin(phi_k) of utils.py:291 (np.linspace(0, 2pi, 50, endpoint=False)), host libm
    double ctab[lsm::kMagSegments], stab[lsm::kMagSegments];
    const double step = (2.0 * lsm::kPi - 0.0) / (double)lsm::kMagSegments;
    for (int k = 0; k < lsm::kMagSegments; ++k) {
        const double phi = (double)k * step + 0.0;
        ctab[k] = lsm_cos(phi); stab[k] = lsm_sin(phi);
    }
    e = lsm::upload_magnetic_tables(ctab, stab);
    if (e != cudaSuccess) { lsm_destroy(h); return cuda_fail(e, "upload_magnetic_tables"); }
    *out = h;
    return 0;
}

int lsm_destroy(lsm_handle* h) {
    if (h == nullptr) return 0;
    DeviceGuard guard(h->device);
    if (h->d_pair_tab) cudaFree(h->d_pair_tab);
    if (h->d_sel_tab) cudaFree(h->d_sel_tab);
    if (h->d_pair32) cudaFree(h->d_pair32);
    if (h->d_pairval) cudaFree(h->d_pairval);
    if (h->d_emit_rec) cudaFree(h->d_emit_rec);
    if (h->d_timeline) cudaFree(h->d_timeline);
    if (h->d_vpacked) cudaFree(h->d_vpacked);
    if (h->d_grads8) cudaFree(h->d_grads8);
    if (h->d_edge_local) cudaFree(h->d_edge_local);
    if (h->d_edge_totals) cudaFree(h->d_edge_totals);
    if (h->d_edge_tickets) cudaFree(h->d_edge_tickets);
    if (h->d_edge_block) cudaFree(h->d_edge_block);
    for (cudaEvent_t ev : h->ev_count) cudaEventDestroy(ev);
    for (cudaStream_t st : h->streams) cudaStreamDestroy(st);
    for (cudaEvent_t ev : h->ev_join) cudaEventDestroy(ev);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    for (cudaEvent_t ev : h->ev_host) cudaEventDestroy(ev);
    if (h->g_exec) cudaGraphExecDestroy(h->g_exec);
    if (h->g_stream) cudaStreamDestroy(h->g_stream);
    std::free(h->g_key); std::free(h->g_seen);
    if (h->d_act) cudaFree(h->d_act);
    if (h->h_act) cudaFreeHost(h->h_act);
    delete h;
    return 0;
}

// Validates the descriptor completely before it touches the handle: a refused grid leaves the bound one (and its packed
// table and padded gradient rows) in place. Every lookup (stencil32_setup, stencil32f_setup, packed_value*, interp_f32)
// forms linear cell indices in int, so grids of 2^31 cells or more are refused.
static int fill_grid(const lsm_grid_desc* g, lsm::GridDev* d, int want_ndim, bool need_grads, const char* who, bool f32) {
    if (g == nullptr || g->values == nullptr) return fail(1, std::string(who) + ": null grid");
    if (g->ndim != want_ndim) return fail(2, std::string(who) + ": wrong grid dimensionality");
    if (need_grads && g->grads == nullptr) return fail(2, std::string(who) + ": gradient array required");
    lsm::GridDev v;
    std::memset(&v, 0, sizeof(v));
    v.ndim = g->ndim;
    unsigned long long cells = 1;
    for (int k = 0; k < g->ndim; ++k) {
        if (g->shape[k] < 2) return fail(2, std::string(who) + ": every grid dimension needs >= 2 nodes");
        cells *= (unsigned long long)g->shape[k];      // < 2^31 before, shape < 2^31: no wrap-around
        if (cells > (unsigned long long)INT_MAX)
            return fail(2, std::string(who) + ": the grid has 2^31 cells or more (32-bit cell indices)");
        v.shape[k] = g->shape[k]; v.periodic[k] = g->periodic[k] ? 1 : 0; v.lo[k] = g->lo[k];
        const double n = (double)g->shape[k];
        v.spacing[k] = g->periodic[k] ? (g->hi[k] - g->lo[k]) / n : (g->hi[k] - g->lo[k]) / (n - 1.0);
        v.inv_spacing[k] = 1.0 / v.spacing[k];
    }
    v.separation_distance = g->separation_distance; v.ttr_max = g->ttr_max;
    v.values = g->values; v.grads = g->grads;
    v.f32 = f32 ? 1 : 0;
    *d = v;
    return 0;
}

int lsm_set_value_grid(lsm_handle* h, const lsm_grid_desc* g) {
    if (h == nullptr) return fail(1, "lsm_set_value_grid: null handle");
    const int want = h->kp.c.dynamics == LSM_DYN_DOUBLE_INTEGRATOR ? 4 : 5;
    int rc = fill_grid(g, &h->kp.vg, want, true, "lsm_set_value_grid", (h->kp.c.flags & LSM_FLAG_INTERP_FLOAT32) != 0);
    if (rc) return rc;
    h->kp.has_vg = 1;
    size_t cells = 1;
    for (int k = 0; k < g->ndim; ++k) cells *= (size_t)g->shape[k];
    // corner-packed copy for the pair kernel (one aligned chunk per lookup; the same table serves the float64 and the
    // float32 lookups); lsm_tuning.packed_grid = 0 keeps the scattered gathers; tables larger than 2 GiB are not built.
    DeviceGuard guard(h->device);
    const bool want_packed = h->tuning.packed_grid != 0;
    if (h->d_vpacked) { cudaFree(h->d_vpacked); h->d_vpacked = nullptr; }
    h->kp.vg.packed = nullptr;
    if (h->spec && want_packed) {
        const size_t max_bytes = (size_t)2048 << 20;
        size_t pcells = 1;      // n slots on periodic dims, n + 1 on the others (see lsm_pack_grid_kernel)
        for (int k = 0; k < g->ndim; ++k) pcells *= (size_t)(g->periodic[k] ? g->shape[k] : g->shape[k] + 1);
        const size_t bytes = pcells * ((size_t)1 << g->ndim) * sizeof(float);
        if (bytes <= max_bytes && pcells < (size_t)0x7fffffff) {
            cudaError_t e = cudaMalloc(&h->d_vpacked, bytes);
            if (e == cudaSuccess) e = lsm::pack_grid_launch(h->kp.vg, h->d_vpacked, (long long)pcells);
            if (e == cudaSuccess) e = cudaDeviceSynchronize();
            if (e != cudaSuccess) return cuda_fail(e, "lsm_set_value_grid: corner-packed table");
            h->kp.vg.packed = h->d_vpacked;
        }
    }
    if (h->d_grads8) { cudaFree(h->d_grads8); h->d_grads8 = nullptr; }
    h->kp.vg.grads8 = nullptr;
    if (h->spec && g->ndim == 5) {     // always: stencil32_grad<5> has no scattered alternative (104 MB for 41x41x24x9x9)
        cudaError_t e = cudaMalloc(&h->d_grads8, cells * 8 * sizeof(float));
        if (e == cudaSuccess) e = lsm::pad_grads_launch(g->grads, h->d_grads8, (long long)cells);
        if (e == cudaSuccess) e = cudaDeviceSynchronize();
        if (e != cudaSuccess) return cuda_fail(e, "lsm_set_value_grid: padded gradient rows");
        h->kp.vg.grads8 = h->d_grads8;
    }
    return 0;
}

int lsm_set_ttr_grid(lsm_handle* h, const lsm_grid_desc* g) {
    if (h == nullptr) return fail(1, "lsm_set_ttr_grid: null handle");
    DeviceGuard guard(h->device);
    int rc = fill_grid(g, &h->kp.tg, 4, false, "lsm_set_ttr_grid", (h->kp.c.flags & LSM_FLAG_INTERP_FLOAT32) != 0);
    if (rc) return rc;
    h->kp.has_tg = 1;
    return 0;
}

int lsm_set_tuning(lsm_handle* h, const lsm_tuning* t) {
    if (h == nullptr || t == nullptr) return fail(1, "lsm_set_tuning: null argument");
    if (t->chunks < 0 || t->chunks > 16) return fail(2, "lsm_set_tuning: chunks must be 0 (automatic) or 1..16");
    if (t->pair_placement != -1 && t->pair_placement != 0 && t->pair_placement != 2 && t->pair_placement != 3 && t->pair_placement != 4)
        return fail(2, "lsm_set_tuning: pair_placement must be -1 (automatic), 0 (behind the emit kernel), 2 (in front of the agent kernel), 3 (between them) or 4 (tail of the agent kernel)");
    if (t->packed_grid < -1 || t->packed_grid > 1) return fail(2, "lsm_set_tuning: packed_grid must be -1, 0 or 1");
    if (t->use_graph < -1 || t->use_graph > 1) return fail(2, "lsm_set_tuning: use_graph must be -1, 0 or 1");
    if (h->have_buffers || h->kp.has_vg) return fail(5, "lsm_set_tuning: call it right after lsm_create (before lsm_set_value_grid / lsm_bind_buffers)");
    h->tuning = *t;
    if (t->pair_placement >= 0) h->pair_placement = t->pair_placement;
    return 0;
}

int lsm_bind_buffers(lsm_handle* h, const lsm_buffers* b) {
    if (h == nullptr || b == nullptr) return fail(1, "lsm_bind_buffers: null argument");
    if (b->num_envs < 1) return fail(2, "lsm_bind_buffers: num_envs must be >= 1");
    const void* ptrs[] = { b->agent_f64, b->agent_i32, b->landmarks, b->env_f64, b->env_i32, b->obs, b->node_obs,
                           b->adj, b->reward, b->done, b->safe_action, b->ep_info };
    for (const void* p : ptrs) if (p == nullptr) return fail(2, "lsm_bind_buffers: every buffer pointer must be non-null");
    if (h->kp.O > 0 && b->obstacles == nullptr) return fail(2, "lsm_bind_buffers: obstacles must be non-null when num_obstacles > 0");
    if (((uintptr_t)b->adj & 15u) || ((uintptr_t)b->node_obs & 15u))
        return fail(2, "lsm_bind_buffers: adj and node_obs must be 16-byte aligned");
    if ((b->term_f64 != nullptr) != (b->term_i32 != nullptr) || (b->term_f64 != nullptr) != (b->term_env_f64 != nullptr))
        return fail(2, "lsm_bind_buffers: term_f64, term_i32 and term_env_f64 must be all set or all NULL");
    DeviceGuard guard(h->device);
    h->kp.b = *b;
    h->kp.adj_base = nullptr; h->kp.adj_keep = nullptr;
    h->kp.edge_index = nullptr;
    h->have_buffers = true;
    // chunked launches for big batches (measured on B200, DESIGN.md 3: 4 ranges pay off from ~0.4 GB of observations per
    // step - 0.8 GB: -11 %, 10.7 GB: -9 % - while a 0.1 GB step is launch-latency bound and stays on the caller's stream:
    // +26 % with 2 ranges). lsm_tuning.chunks overrides.
    {
        const double step_bytes = (double)b->num_envs * 4.0 * h->kp.N * h->kp.E * (double)(h->kp.F + h->kp.E);
        int want = step_bytes >= 4.0e8 ? 4 : 1;
        if (h->tuning.chunks >= 1 && h->tuning.chunks <= 16) want = h->tuning.chunks;
        if (!h->spec) want = 1;
        h->chunks = want;
        while ((int)h->streams.size() < (want > 1 ? want : 0)) {
            cudaStream_t st; cudaEvent_t ev;
            cudaError_t e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
            if (e != cudaSuccess) return cuda_fail(e, "lsm_bind_buffers: chunk streams");
            h->streams.push_back(st); h->ev_join.push_back(ev);
        }
        if (want > 1 && h->ev_fork == nullptr) {
            cudaError_t e = cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming);
            if (e != cudaSuccess) return cuda_fail(e, "lsm_bind_buffers: chunk streams");
        }
    }
    if (h->d_edge_local) { cudaFree(h->d_edge_local); h->d_edge_local = nullptr; }     // sized by num_envs: re-made on demand
    if (h->d_edge_totals) { cudaFree(h->d_edge_totals); h->d_edge_totals = nullptr; }
    if (h->d_edge_tickets) { cudaFree(h->d_edge_tickets); h->d_edge_tickets = nullptr; }
    if (h->d_edge_block) { cudaFree(h->d_edge_block); h->d_edge_block = nullptr; }
    if (h->spec) {
        // library-owned scratch between the launches of one step
        if (h->d_pairval) { cudaFree(h->d_pairval); h->d_pairval = nullptr; }
        if (h->d_emit_rec) { cudaFree(h->d_emit_rec); h->d_emit_rec = nullptr; }
        const size_t N = (size_t)h->kp.N;
        cudaError_t e = cudaMalloc(&h->d_pairval, (size_t)b->num_envs * N * N * sizeof(double));
        if (e == cudaSuccess) e = cudaMalloc(&h->d_emit_rec, (size_t)b->num_envs * (size_t)h->tab.rec_bytes);
        if (e != cudaSuccess) return cuda_fail(e, "lsm_bind_buffers: scratch allocation");
        h->kp.emit_rec = h->d_emit_rec;
        h->pairval_valid = false;
    }
    return 0;
}

int lsm_get_launch_info(lsm_handle* h, lsm_launch_info* out) {
    if (h == nullptr || out == nullptr) return fail(1, "lsm_get_launch_info: null argument");
    const long long ngroups = h->have_buffers ? (h->kp.b.num_envs + h->kp.EPW - 1) / h->kp.EPW : 0;
    long long blocks = (ngroups + h->warps_per_block - 1) / h->warps_per_block;
    if (!h->spec && blocks > h->grid_cap) blocks = h->grid_cap;
    out->grid_blocks = (int32_t)blocks; out->block_threads = h->block_threads; out->warps_per_block = h->warps_per_block;
    out->envs_per_warp = h->kp.EPW; out->smem_bytes_per_block = h->smem_per_block; out->regs_per_thread = h->regs;
    out->blocks_per_sm = h->blocks_per_sm; out->sm_count = h->sm_count;
    out->specialised = h->spec ? 1 : 0;
    out->emit_block_threads = h->tab.emit_threads;
    out->emit_smem_bytes_per_block = h->tab.emit_smem;
    out->emit_regs_per_thread = h->tab.emit_regs; out->emit_blocks_per_sm = h->tab.emit_blocks_per_sm;
    const bool pair_path_li = h->spec && (h->kp.c.flags & LSM_FLAG_USE_SAFETY_FILTER) && h->kp.has_vg;
    out->pair_regs_per_thread = h->tab.pair_regs;
    out->launches_per_step = h->spec ? ((pair_path_li && h->pair_placement != 4) ? 3 : 2) : 1;   // agent, emit [, pair]
    out->emit_record_bytes = h->tab.rec_bytes;
    {
        const int K = (h->spec && h->chunks > 1 && ngroups >= 4LL * h->chunks * h->warps_per_block) ? h->chunks : 1;
        out->chunks = K;
        out->launches_per_step *= K;
        out->pair_placement = pair_path_li ? h->pair_placement : -1;
    }
    out->graph_replays = (int32_t)std::min<long long>(h->g_replays, 0x7fffffff);
    out->graph_captures = (int32_t)std::min<long long>(h->g_captures, 0x7fffffff);
    return 0;
}

static int launch(lsm_handle* h, int mode, int flag, const int32_t* action_idx, const float* action_onehot,
                  const uint8_t* env_mask, int64_t episode, uint64_t seed, void* stream, const char* who) {
    if (h == nullptr) return fail(1, std::string(who) + ": null handle");
    if (!h->have_buffers) return fail(5, std::string(who) + ": lsm_bind_buffers has not been called");
    const lsm_config& c = h->kp.c;
    const bool needs_vg = (c.flags & (LSM_FLAG_USE_SAFETY_FILTER | LSM_FLAG_HJ_VALUE)) != 0;
    if (needs_vg && !h->kp.has_vg) return fail(5, std::string(who) + ": safety filter / HJ_VALUE enabled but no value grid set");
    if (c.dynamics == LSM_DYN_AIRTAXI && !h->kp.has_tg) return fail(5, std::string(who) + ": airtaxi needs a TTR grid");
    lsm::KParams kp = h->kp;
    kp.mode = mode; kp.flag = flag; kp.action_idx = action_idx; kp.action_onehot = action_onehot;
    kp.env_mask = env_mask; kp.episode = (long long)episode; kp.seed = (unsigned long long)seed;
    const long long ngroups = (kp.b.num_envs + kp.EPW - 1) / kp.EPW;
    DeviceGuard guard(h->device);
    const bool pair_path = h->spec && (c.flags & LSM_FLAG_USE_SAFETY_FILTER) && h->kp.has_vg;
    const int placement = h->pair_placement;
    const bool was_valid = h->pairval_valid;

    const bool edges = h->spec && kp.edge_index != nullptr;
    // the agent kernel of this launch writes the emit record of every env of its range (a masked reset only those in
    // the mask): the pair kernel behind it can then read its inputs from the records (see lsm_pair_kernel)
    const bool rec_fresh = !(mode == lsm::MODE_RESET && env_mask != nullptr);
    // the launches of one env-group range [g0, g1) on stream `s` (range `q` of `nq`)
    auto launch_range = [&](long long g0, long long g1, cudaStream_t s, int q, int nq) -> cudaError_t {
        lsm::KParams k = kp;
        k.edge_range = q; k.edge_num_ranges = nq;
        if (edges) {
            // count blocks take contiguous runs of environments; every range owns a slice of the block arrays
            const long long per_range_envs = (long long)kp.EPW * (((ngroups + nq - 1) / nq + h->warps_per_block - 1) / h->warps_per_block * h->warps_per_block);
            k.edge_envs_per_block = lsm::edge_count_envs_per_block(nq > 1 ? per_range_envs : kp.b.num_envs);
            k.edge_block_ofs = (int)(q * ((per_range_envs + k.edge_envs_per_block - 1) / k.edge_envs_per_block + 1));
        }
        k.grp_begin = (int)g0; k.ngroups = (int)g1;
        k.env_begin = (int)(g0 * kp.EPW);
        k.env_end = (int)std::min<long long>(kp.b.num_envs, g1 * kp.EPW);
        long long blocks = (g1 - g0 + h->warps_per_block - 1) / h->warps_per_block;
        if (!h->spec && blocks > h->grid_cap) blocks = h->grid_cap;   // generic kernel: persistent grid
        cudaError_t e;
        k.pairval = nullptr;
        k.pair_late = 0;
        k.pair_tail = 0;
        k.pair_rec = 0;
        if (pair_path && placement == 4) {
            // the agent kernel leaves the next step's pair values behind itself (all modes: a reset / observe launch makes
            // them valid for the step that follows)
            k.pairval = h->d_pairval;
            k.pair_tail = 1;
        }
        if (pair_path && mode == lsm::MODE_STEP) {
            // HJ values of every ordered agent pair for the states this step starts from: normally left behind by the
            // previous launch (emit kernel / late pair kernel); recomputed here when the state was edited in between
            k.pairval = h->d_pairval;
            if (!was_valid || placement == 2) {
                e = lsm::spec_launch_pair(k, h->tab, h->sm_count, s);
                if (e != cudaSuccess) return e;
            }
        }
        // K_b (specialised: per-agent physics) or the fused generic kernel
        e = lsm::kernel_launch(h->spec ? h->tab.agent : lsm::generic_ptr(c.dynamics), k, (unsigned)blocks, h->block_threads,
                               h->smem_per_block, s, h->spec);
        if (e != cudaSuccess) return e;
        if (h->spec) {
            if (pair_path && placement == 3) {
                // K_a for the NEXT step between the agent and the emit kernel: alone on the GPU at full occupancy
                k.pairval = h->d_pairval;
                k.pair_late = 0;
                k.pair_rec = rec_fresh ? 1 : 0;
                e = lsm::spec_launch_pair(k, h->tab, h->sm_count, s);
                k.pair_rec = 0;
                if (e != cudaSuccess) return e;
            }
            if (edges) {
                // fused COO output: where every graph's edges start (counts + prefix inside this range); the emit kernel of
                // a later range also needs the totals of the earlier ones -> ordered by events, never by spinning
                k.pairval = nullptr;
                e = lsm::spec_launch_edge_count(k, h->tab, s);
                if (e != cudaSuccess) return e;
                if (nq > 1) {
                    if ((e = cudaEventRecord(h->ev_count[q], s)) != cudaSuccess) return e;
                    for (int r = 0; r < q; ++r)
                        if ((e = cudaStreamWaitEvent(s, h->ev_count[r], 0)) != cudaSuccess) return e;
                }
            }
            // K_c: graph observation (persistent blocks)
            k.pairval = nullptr;
            e = lsm::spec_launch_emit(k, h->tab, h->sm_count, s);
            if (e != cudaSuccess) return e;
            if (pair_path && placement == 0) {
                // K_a for the NEXT step, beside the emit kernel's drain (see lsm_pair_kernel)
                k.pairval = h->d_pairval;
                k.pair_late = 1;
                k.pair_rec = rec_fresh ? 1 : 0;
                e = lsm::spec_launch_pair(k, h->tab, h->sm_count, s);
                if (e != cudaSuccess) return e;
            }
        }
        return cudaSuccess;
    };

    cudaError_t e = cudaSuccess;
    const int K = (h->spec && h->chunks > 1 && ngroups >= 4LL * h->chunks * h->warps_per_block) ? h->chunks : 1;
    // graph replay: single-range steps of the specialised pipeline (the launch-latency-bound sizes); opt-in - measured on
    // B200 it cuts the host time of a step from ~25 to ~9 us but adds ~1 us of device time (DESIGN.md 3)
    bool use_graph = h->spec && K == 1 && mode == lsm::MODE_STEP && h->tuning.use_graph == 1 && kp.timeline == nullptr;
    if (use_graph) {
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing((cudaStream_t)stream, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) {
            (void)cudaGetLastError();
            use_graph = false;              // the caller is capturing this stream itself: plain launches join its graph
        }
    }
    if (use_graph) {
        typedef lsm_handle::GraphKey GK;
        if (h->g_key == nullptr) {
            h->g_key = (GK*)std::calloc(1, sizeof(GK)); h->g_seen = (GK*)std::calloc(1, sizeof(GK));
            if (h->g_key == nullptr || h->g_seen == nullptr) return fail(4, std::string(who) + ": out of host memory");
        }
        static thread_local GK cur;         // compared bytewise: build it in zeroed storage
        std::memset(&cur, 0, sizeof(cur));
        std::memcpy(&cur.kp, &kp, sizeof(kp)); cur.was_valid = was_valid ? 1 : 0; cur.placement = placement;
        bool replay = h->g_exec != nullptr && h->g_key_valid && std::memcmp(&cur, h->g_key, sizeof(GK)) == 0;
        if (!replay && h->g_seen_valid && std::memcmp(&cur, h->g_seen, sizeof(GK)) == 0) {
            // second launch in a row with these parameters: capture it
            if (h->g_stream == nullptr && (e = cudaStreamCreateWithFlags(&h->g_stream, cudaStreamNonBlocking)) != cudaSuccess)
                return cuda_fail(e, who);
            cudaGraph_t graph = nullptr;
            e = cudaStreamBeginCapture(h->g_stream, cudaStreamCaptureModeThreadLocal);
            if (e == cudaSuccess) {
                const cudaError_t el = launch_range(0, ngroups, h->g_stream, 0, 1);
                e = cudaStreamEndCapture(h->g_stream, &graph);
                if (el != cudaSuccess) e = el;
            }
            if (e == cudaSuccess && h->g_exec != nullptr) {
                cudaGraphExecUpdateResultInfo info;
                if (cudaGraphExecUpdate(h->g_exec, graph, &info) != cudaSuccess) {
                    (void)cudaGetLastError();
                    cudaGraphExecDestroy(h->g_exec); h->g_exec = nullptr;
                }
            }
            if (e == cudaSuccess && h->g_exec == nullptr) e = cudaGraphInstantiate(&h->g_exec, graph, 0);
            if (graph) cudaGraphDestroy(graph);
            if (e == cudaSuccess) {
                std::memcpy(h->g_key, &cur, sizeof(GK)); h->g_key_valid = true; ++h->g_captures;
                replay = true;
            } else {
                // capture is an optimisation: fall back to the plain launches for the rest of this handle's life
                (void)cudaGetLastError();
                if (h->g_exec) { cudaGraphExecDestroy(h->g_exec); h->g_exec = nullptr; }
                h->g_key_valid = false; h->tuning.use_graph = 0;
            }
        }
        if (replay) {
            if ((e = cudaGraphLaunch(h->g_exec, (cudaStream_t)stream)) != cudaSuccess) return cuda_fail(e, who);
            ++h->g_replays;
        } else {
            std::memcpy(h->g_seen, &cur, sizeof(GK)); h->g_seen_valid = true;
            e = launch_range(0, ngroups, (cudaStream_t)stream, 0, 1);
            if (e != cudaSuccess) return cuda_fail(e, who);
        }
    } else if (K == 1) {
        e = launch_range(0, ngroups, (cudaStream_t)stream, 0, 1);
        if (e != cudaSuccess) return cuda_fail(e, who);
    } else {
        // fork: every library stream waits for the caller's stream; join: the caller's stream waits for every range
        if ((e = cudaEventRecord(h->ev_fork, (cudaStream_t)stream)) != cudaSuccess) return cuda_fail(e, who);
        const long long per = ((ngroups + K - 1) / K + h->warps_per_block - 1) / h->warps_per_block * h->warps_per_block;
        for (int q = 0; q < K; ++q) {
            const long long g0 = std::min<long long>(ngroups, per * q), g1 = std::min<long long>(ngroups, per * (q + 1));
            if (g0 >= g1) continue;
            if ((e = cudaStreamWaitEvent(h->streams[q], h->ev_fork, 0)) != cudaSuccess) return cuda_fail(e, who);
            if ((e = launch_range(g0, g1, h->streams[q], q, K)) != cudaSuccess) return cuda_fail(e, who);
            if ((e = cudaEventRecord(h->ev_join[q], h->streams[q])) != cudaSuccess) return cuda_fail(e, who);
            if ((e = cudaStreamWaitEvent((cudaStream_t)stream, h->ev_join[q], 0)) != cudaSuccess) return cuda_fail(e, who);
        }
    }
    if (h->spec) {
        h->pairval_valid = false;
        if (pair_path && (placement == 0 || placement == 3)) h->pairval_valid = true;
        // placement 4: a masked reset refreshes only the masked environments, the others keep what they had
        if (pair_path && placement == 4)
            h->pairval_valid = env_mask == nullptr ? true : (was_valid && mode != lsm::MODE_STEP);
    }
    return 0;
}

int lsm_step(lsm_handle* h, const int32_t* action_idx, const float* action_onehot, int64_t episode, uint64_t seed,
             int auto_reset, void* stream) {
    if ((action_idx == nullptr) == (action_onehot == nullptr))
        return fail(2, "lsm_step: pass exactly one of action_idx / action_onehot");
    return launch(h, lsm::MODE_STEP, auto_reset ? 1 : 0, action_idx, action_onehot, nullptr, episode, seed, stream, "lsm_step");
}

int lsm_reset(lsm_handle* h, const uint8_t* env_mask, int64_t episode, uint64_t seed, int sample, void* stream) {
    return launch(h, lsm::MODE_RESET, sample ? 1 : 0, nullptr, nullptr, env_mask, episode, seed, stream, "lsm_reset");
}

int lsm_observe(lsm_handle* h, void* stream) {
    return launch(h, lsm::MODE_OBSERVE, 0, nullptr, nullptr, nullptr, 0, 0, stream, "lsm_observe");
}

int lsm_set_output_buffers(lsm_handle* h, float* obs, float* node_obs, float* adj, float* reward, uint8_t* done) {
    if (h == nullptr) return fail(1, "lsm_set_output_buffers: null handle");
    if (!h->have_buffers) return fail(5, "lsm_set_output_buffers: lsm_bind_buffers has not been called");
    if (((uintptr_t)adj & 15u) || ((uintptr_t)node_obs & 15u))
        return fail(2, "lsm_set_output_buffers: adj and node_obs must be 16-byte aligned");
    if (obs) h->kp.b.obs = obs;
    if (node_obs) h->kp.b.node_obs = node_obs;
    if (adj) h->kp.b.adj = adj;
    if (reward) h->kp.b.reward = reward;
    if (done) h->kp.b.done = done;
    return 0;
}

int lsm_set_compact_adjacency(lsm_handle* h, float* adj_base, uint32_t* adj_keep) {
    if (h == nullptr) return fail(1, "lsm_set_compact_adjacency: null handle");
    if (!h->have_buffers) return fail(5, "lsm_set_compact_adjacency: lsm_bind_buffers has not been called");
    if ((adj_base == nullptr) != (adj_keep == nullptr)) return fail(2, "lsm_set_compact_adjacency: pass both pointers or neither");
    if (adj_base != nullptr && !h->spec)
        return fail(6, "lsm_set_compact_adjacency: this configuration runs the fused generic kernel (dense adjacency only)");
    if ((uintptr_t)adj_base & 15u) return fail(2, "lsm_set_compact_adjacency: adj_base must be 16-byte aligned");
    h->kp.adj_base = adj_base; h->kp.adj_keep = adj_keep;
    return 0;
}

// entities of the largest environment lsm_create accepts (agents + landmarks + obstacles), rounded up to the 4-float
// steps of the vector path: the host expansion's per-row buffers hold this many entries
constexpr int kMaxEntities = LSM_MAX_AGENTS + LSM_MAX_LANDMARKS + LSM_MAX_OBSTACLES;
constexpr int kRowCap = (kMaxEntities + 3) / 4 * 4;

// one environment range of the host-side adjacency expansion (pure data movement: every float is copied or zero)
static void expand_adjacency_range(const float* adj_base, const uint32_t* adj_keep, float* adj, int64_t e0, int64_t e1, int N, int E,
                                   bool cached_stores) {
    const int W = (E + 31) / 32, EE = E * E;
    const bool vec = (EE % 4) == 0;          // every observer matrix starts 16-byte aligned
    alignas(16) float row[kRowCap];
    for (int64_t e = e0; e < e1; ++e) {
        const float* base = adj_base + e * EE;
        for (int i = 0; i < N; ++i) {
            const uint32_t* keep = adj_keep + (e * N + i) * W;
            float* dst = adj + (e * N + i) * EE;
            if (vec && (E % 4) == 0) {
                bool all = true;
                for (int w = 0; w < W; ++w) {
                    const uint32_t full = (w == W - 1 && (E & 31)) ? ((1u << (E & 31)) - 1u) : 0xffffffffu;
                    all = all && ((keep[w] & full) == full);
                }
                if (all) {
                    // nothing is disconnected for this observer (the common case): a straight streaming copy
                    const __m128i* s4 = (const __m128i*)base; __m128i* d4 = (__m128i*)dst;
                    if (cached_stores) for (int q = 0; q < EE / 4; ++q) _mm_store_si128(d4 + q, _mm_loadu_si128(s4 + q));
                    else for (int q = 0; q < EE / 4; ++q) _mm_stream_si128(d4 + q, _mm_loadu_si128(s4 + q));
                    continue;
                }
                // rows are 16-byte multiples: build the column mask once per observer, stream the rows
                alignas(16) uint32_t cm[kRowCap];
                for (int b = 0; b < E; ++b) cm[b] = ((keep[b >> 5] >> (b & 31)) & 1u) ? 0xffffffffu : 0u;
                for (int a = 0; a < E; ++a) {
                    const bool ka = (keep[a >> 5] >> (a & 31)) & 1u;
                    const __m128i am = _mm_set1_epi32(ka ? -1 : 0);
                    for (int b = 0; b < E; b += 4) {
                        const __m128i v = _mm_loadu_si128((const __m128i*)(base + a * E + b));
                        const __m128i m = _mm_and_si128(_mm_load_si128((const __m128i*)(cm + b)), am);
                        if (cached_stores) _mm_store_si128((__m128i*)(dst + a * E + b), _mm_and_si128(v, m));
                        else _mm_stream_si128((__m128i*)(dst + a * E + b), _mm_and_si128(v, m));
                    }
                }
            } else {
                for (int a = 0; a < E; ++a) {
                    const bool ka = (keep[a >> 5] >> (a & 31)) & 1u;
                    for (int b = 0; b < E; ++b) {
                        const bool kb = (keep[b >> 5] >> (b & 31)) & 1u;
                        row[b] = (ka && kb) ? base[a * E + b] : 0.0f;
                    }
                    std::memcpy(dst + a * E, row, sizeof(float) * E);
                }
            }
        }
    }
    _mm_sfence();
}

static int resolve_host_threads(int threads, int64_t num_envs) {
    int T = threads;
    if (T <= 0) { T = (int)std::thread::hardware_concurrency(); if (T < 1) T = 1; if (T > 16) T = 16; }
    if (T > 64) T = 64;
    if ((int64_t)T > num_envs) T = (int)num_envs;
    return T < 1 ? 1 : T;
}

int lsm_expand_adjacency_host(const float* adj_base, const uint32_t* adj_keep, float* adj, int64_t num_envs, int32_t N, int32_t E,
                              int32_t threads, int32_t cached_stores) {
    if (adj_base == nullptr || adj_keep == nullptr || adj == nullptr) return fail(1, "lsm_expand_adjacency_host: null argument");
    if (num_envs < 0 || N < 1 || N > LSM_MAX_AGENTS || E < N || E > kMaxEntities)
        return fail(2, "lsm_expand_adjacency_host: bad sizes");
    if (((uintptr_t)adj & 3u) || (((E * E) % 4) == 0 && ((uintptr_t)adj & 15u)))
        return fail(2, "lsm_expand_adjacency_host: adj must be 16-byte aligned (4-byte when E*E is not a multiple of 4)");
    if (num_envs == 0) return 0;
    const int T = resolve_host_threads(threads, num_envs);
    auto work = [&](int part) {
        expand_adjacency_range(adj_base, adj_keep, adj, num_envs * part / T, num_envs * (part + 1) / T, N, E, cached_stores != 0);
    };
    if (T == 1) work(0);
    else HostPool::get().run(T, work);
    return 0;
}

// D2H of one step's outputs + host expansion of the compact adjacency, pipelined: the compact matrices leave first in
// `chunks` env ranges with an event behind each; the calling thread waits for the events in order and publishes
// "range c has landed", the pool's workers expand the ranges as they land while the DMA engine is still moving the
// later ranges and node_obs. Returns when every host array is complete.
int lsm_fetch_host(lsm_handle* h, const lsm_host_io* io, void* stream) {
    if (h == nullptr || io == nullptr) return fail(1, "lsm_fetch_host: null argument");
    if (!h->have_buffers) return fail(5, "lsm_fetch_host: lsm_bind_buffers has not been called");
    if (h->kp.adj_base == nullptr) return fail(5, "lsm_fetch_host: needs the compact adjacency (lsm_set_compact_adjacency)");
    if (io->adj == nullptr || io->adj_base_staging == nullptr || io->adj_keep_staging == nullptr)
        return fail(2, "lsm_fetch_host: adj, adj_base_staging and adj_keep_staging are required");
    const int N = h->kp.N, E = h->kp.E, W = (E + 31) / 32, EE = E * E;
    if (E > kMaxEntities) return fail(2, "lsm_fetch_host: more entities than the host expansion holds");
    if (((uintptr_t)io->adj & 3u) || ((EE % 4) == 0 && ((uintptr_t)io->adj & 15u)))
        return fail(2, "lsm_fetch_host: adj must be 16-byte aligned (4-byte when E*E is not a multiple of 4)");
    const int64_t n = h->kp.b.num_envs;
    DeviceGuard guard(h->device);
    cudaStream_t s = (cudaStream_t)stream;
    int Cn = io->chunks > 0 ? io->chunks : (n >= 2048 ? 8 : (n >= 256 ? 4 : 1));
    if (Cn > 64) Cn = 64;
    if ((int64_t)Cn > n) Cn = (int)n;
    while ((int)h->ev_host.size() < Cn + 1) {
        cudaEvent_t ev;
        cudaError_t e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
        if (e != cudaSuccess) return cuda_fail(e, "lsm_fetch_host: events");
        h->ev_host.push_back(ev);
    }
    cudaError_t e = cudaSuccess;
    for (int c = 0; c < Cn && e == cudaSuccess; ++c) {
        const int64_t lo = n * c / Cn, hi = n * (c + 1) / Cn;
        e = cudaMemcpyAsync(io->adj_base_staging + lo * EE, h->kp.adj_base + lo * EE, (size_t)(hi - lo) * EE * sizeof(float), cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(io->adj_keep_staging + lo * N * W, h->kp.adj_keep + lo * N * W, (size_t)(hi - lo) * N * W * sizeof(uint32_t), cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaEventRecord(h->ev_host[c], s);
    }
    const bool gfeat = (h->kp.c.flags & LSM_FLAG_GRAPH_FEAT_GLOBAL) != 0;
    const size_t Fr = gfeat ? 7 : (size_t)h->kp.F;
    if (e == cudaSuccess && io->obs) e = cudaMemcpyAsync(io->obs, h->kp.b.obs, (size_t)n * N * h->kp.D * sizeof(float), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess && io->reward) e = cudaMemcpyAsync(io->reward, h->kp.b.reward, (size_t)n * N * sizeof(float), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess && io->done) e = cudaMemcpyAsync(io->done, h->kp.b.done, (size_t)n * N, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess && io->node_obs) e = cudaMemcpyAsync(io->node_obs, h->kp.b.node_obs, (size_t)n * N * E * Fr * sizeof(float), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaEventRecord(h->ev_host[Cn], s);
    if (e != cudaSuccess) return cuda_fail(e, "lsm_fetch_host: enqueue");

    const int T = resolve_host_threads(io->threads, n);
    const int P = T;                                  // parts per range: every worker gets a share of every range
    std::atomic<int> ready{0}, next{0};
    std::atomic<int> err{0};
    const bool cached = io->cached_stores != 0;
    auto drain = [&]() {
        for (;;) {
            const int item = next.fetch_add(1, std::memory_order_relaxed);
            if (item >= Cn * P) return;
            const int c = item / P, p = item - c * P;
            while (ready.load(std::memory_order_acquire) <= c) _mm_pause();
            if (err.load(std::memory_order_relaxed)) continue;
            const int64_t lo = n * c / Cn, hi = n * (c + 1) / Cn;
            const int64_t e0 = lo + (hi - lo) * p / P, e1 = lo + (hi - lo) * (p + 1) / P;
            expand_adjacency_range(io->adj_base_staging, io->adj_keep_staging, io->adj, e0, e1, N, E, cached);
        }
    };
    auto work = [&](int part) {
        if (part == 0) {
            for (int c = 0; c < Cn; ++c) {
                const cudaError_t ee = cudaEventSynchronize(h->ev_host[c]);
                if (ee != cudaSuccess) { err.store((int)ee); ready.store(Cn, std::memory_order_release); break; }
                ready.store(c + 1, std::memory_order_release);
            }
        }
        drain();
    };
    if (T == 1) work(0);
    else HostPool::get().run(T, work);
    if (err.load()) return cuda_fail((cudaError_t)err.load(), "lsm_fetch_host: waiting for the adjacency ranges");
    e = cudaEventSynchronize(h->ev_host[Cn]);
    if (e != cudaSuccess) return cuda_fail(e, "lsm_fetch_host: waiting for the copies");
    return 0;
}

// The whole reference-facing step with HOST buffers in one call (GraphSubprocVecEnv.step, env_wrappers.py:951-996): actions
// host -> device, the step's launches, outputs device -> host (lsm_fetch_host).
int lsm_step_host(lsm_handle* h, const int32_t* action_idx_host, const float* action_onehot_host, int64_t episode, uint64_t seed,
                  int auto_reset, const lsm_host_io* io, void* stream) {
    if (h == nullptr || io == nullptr) return fail(1, "lsm_step_host: null argument");
    if ((action_idx_host == nullptr) == (action_onehot_host == nullptr))
        return fail(2, "lsm_step_host: pass exactly one of action_idx_host / action_onehot_host");
    if (!h->have_buffers) return fail(5, "lsm_step_host: lsm_bind_buffers has not been called");
    const int64_t n = h->kp.b.num_envs;
    const size_t bytes = action_idx_host ? (size_t)n * h->kp.N * sizeof(int32_t) : (size_t)n * h->kp.N * LSM_NUM_ACTIONS * sizeof(float);
    const void* src = action_idx_host ? (const void*)action_idx_host : (const void*)action_onehot_host;
    cudaStream_t s = (cudaStream_t)stream;
    {
        DeviceGuard guard(h->device);
        cudaError_t e = cudaSuccess;
        if (h->act_bytes < bytes) {
            if (h->d_act) cudaFree(h->d_act);
            if (h->h_act) cudaFreeHost(h->h_act);
            h->d_act = nullptr; h->h_act = nullptr; h->act_bytes = 0;
            e = cudaMalloc(&h->d_act, bytes);
            if (e == cudaSuccess) e = cudaHostAlloc(&h->h_act, bytes, cudaHostAllocDefault);
            if (e != cudaSuccess) return cuda_fail(e, "lsm_step_host: action staging");
            h->act_bytes = bytes;
        }
        // page-locked caller memory is DMA'd in place; pageable memory goes through the library's pinned staging buffer
        // (the previous step's copy out of it has completed: every lsm_step_host ends with a stream-ordered host wait)
        cudaPointerAttributes attr;
        const bool pinned = cudaPointerGetAttributes(&attr, src) == cudaSuccess && attr.type == cudaMemoryTypeHost;
        (void)cudaGetLastError();
        if (!pinned) { std::memcpy(h->h_act, src, bytes); src = h->h_act; }
        e = cudaMemcpyAsync(h->d_act, src, bytes, cudaMemcpyHostToDevice, s);
        if (e != cudaSuccess) return cuda_fail(e, "lsm_step_host: action copy");
    }
    int rc = lsm_step(h, action_idx_host ? (const int32_t*)h->d_act : nullptr, action_onehot_host ? (const float*)h->d_act : nullptr,
                      episode, seed, auto_reset, stream);
    if (rc) return rc;
    return lsm_fetch_host(h, io, stream);
}

int lsm_set_edge_output(lsm_handle* h, int64_t* edge_index, float* edge_attr, int32_t* counts, int64_t* offsets, int64_t capacity,
                        int dense_adj) {
    if (h == nullptr) return fail(1, "lsm_set_edge_output: null handle");
    if (!h->have_buffers) return fail(5, "lsm_set_edge_output: lsm_bind_buffers has not been called");
    if (edge_index == nullptr && edge_attr == nullptr && counts == nullptr && offsets == nullptr) { h->kp.edge_index = nullptr; return 0; }
    if (edge_index == nullptr || edge_attr == nullptr || counts == nullptr || offsets == nullptr)
        return fail(2, "lsm_set_edge_output: pass all four arrays, or all NULL to switch the edge output off");
    if (capacity < 1) return fail(2, "lsm_set_edge_output: capacity must be >= 1");
    if (!h->spec) return fail(6, "lsm_set_edge_output: this configuration runs the fused generic kernel (use lsm_edge_list on the dense adjacency)");
    if (h->kp.adj_base != nullptr && dense_adj) return fail(2, "lsm_set_edge_output: dense_adj is not available together with the compact adjacency");
    DeviceGuard guard(h->device);
    cudaError_t e = cudaSuccess;
    const size_t graphs = (size_t)h->kp.b.num_envs * (size_t)h->kp.N;
    if (h->d_edge_local == nullptr) {
        // count blocks of one step: <= num_envs / 4 + one per env range
        h->edge_block_cap = (size_t)h->kp.b.num_envs / 4 + 64;
        e = cudaMalloc(&h->d_edge_local, graphs * sizeof(int));
        if (e == cudaSuccess) e = cudaMalloc(&h->d_edge_block, 2 * h->edge_block_cap * sizeof(long long));
        if (e == cudaSuccess) e = cudaMalloc(&h->d_edge_totals, 16 * sizeof(long long));
        if (e == cudaSuccess) e = cudaMalloc(&h->d_edge_tickets, 16 * sizeof(unsigned));
        if (e == cudaSuccess) e = cudaMemset(h->d_edge_totals, 0, 16 * sizeof(long long));
        if (e == cudaSuccess) e = cudaMemset(h->d_edge_tickets, 0, 16 * sizeof(unsigned));
        if (e != cudaSuccess) return cuda_fail(e, "lsm_set_edge_output: scratch allocation");
    }
    while ((int)h->ev_count.size() < 16) {
        cudaEvent_t ev;
        if ((e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess) return cuda_fail(e, "lsm_set_edge_output: events");
        h->ev_count.push_back(ev);
    }
    h->kp.edge_index = (long long*)edge_index; h->kp.edge_attr = edge_attr; h->kp.edge_counts = counts;
    h->kp.edge_offsets = (long long*)offsets; h->kp.edge_capacity = (long long)capacity; h->kp.edge_dense = dense_adj ? 1 : 0;
    h->kp.edge_local = h->d_edge_local; h->kp.edge_range_totals = h->d_edge_totals; h->kp.edge_tickets = h->d_edge_tickets;
    h->kp.edge_block_totals = h->d_edge_block; h->kp.edge_block_base = h->d_edge_block + h->edge_block_cap;
    return 0;
}

int lsm_edge_list(lsm_handle* h, const float* adj, int64_t* edge_index, float* edge_attr, int32_t* counts, int64_t* offsets,
                  int64_t capacity, void* stream) {
    if (h == nullptr) return fail(1, "lsm_edge_list: null handle");
    if (!h->have_buffers) return fail(5, "lsm_edge_list: lsm_bind_buffers has not been called");
    if (edge_index == nullptr || edge_attr == nullptr || counts == nullptr || offsets == nullptr)
        return fail(1, "lsm_edge_list: null output");
    if (capacity < 1) return fail(2, "lsm_edge_list: capacity must be >= 1");
    DeviceGuard guard(h->device);
    const float* a = adj ? adj : h->kp.b.adj;
    const long long graphs = (long long)h->kp.b.num_envs * h->kp.N;
    cudaError_t e = lsm::edge_list_launch(a, counts, (long long*)offsets, (long long*)edge_index, edge_attr, graphs, h->kp.E,
                                          (long long)capacity, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "lsm_edge_list");
    return 0;
}

int lsm_world_graph(lsm_handle* h, int64_t* edge_index, double* edge_weight, int32_t* counts, int64_t* offsets, int64_t capacity,
                    void* stream) {
    if (h == nullptr) return fail(1, "lsm_world_graph: null handle");
    if (!h->have_buffers) return fail(5, "lsm_world_graph: lsm_bind_buffers has not been called");
    if (edge_index == nullptr || edge_weight == nullptr || counts == nullptr || offsets == nullptr)
        return fail(1, "lsm_world_graph: null output");
    if (capacity < 1) return fail(2, "lsm_world_graph: capacity must be >= 1");
    DeviceGuard guard(h->device);
    cudaError_t e = lsm::world_graph_launch(h->kp, counts, (long long*)offsets, (long long*)edge_index, edge_weight, (long long)capacity,
                                            (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "lsm_world_graph");
    return 0;
}

int lsm_rollout_insert(lsm_handle* h, const float* obs, const uint8_t* done, float* share_obs, float* masks, float* active_masks,
                       void* stream) {
    if (h == nullptr) return fail(1, "lsm_rollout_insert: null handle");
    if (!h->have_buffers) return fail(5, "lsm_rollout_insert: lsm_bind_buffers has not been called");
    if (obs == nullptr || done == nullptr || masks == nullptr || active_masks == nullptr)
        return fail(1, "lsm_rollout_insert: obs, done, masks and active_masks must be non-null");
    DeviceGuard guard(h->device);
    cudaError_t e = lsm::rollout_insert_launch(obs, done, share_obs, masks, active_masks, (long long)h->kp.b.num_envs, h->kp.N, h->kp.D,
                                               (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "lsm_rollout_insert");
    return 0;
}

int lsm_episode_stats(lsm_handle* h, double* out, void* stream) {
    if (h == nullptr || out == nullptr) return fail(1, "lsm_episode_stats: null argument");
    if (!h->have_buffers) return fail(5, "lsm_episode_stats: lsm_bind_buffers has not been called");
    DeviceGuard guard(h->device);
    cudaError_t e = lsm::episode_stats_launch(h->kp.b.ep_info, (long long)h->kp.b.num_envs, out, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "lsm_episode_stats");
    return 0;
}

int lsm_math_eval(int op, const double* a, const double* b, double* out, int64_t n) {
    if (a == nullptr || out == nullptr || (op == 2 && b == nullptr)) return fail(1, "lsm_math_eval: null argument");
    if (op < 0 || op > 4) return fail(2, "lsm_math_eval: op must be 0 sin, 1 cos, 2 atan2, 3 sincos.sin, 4 sincos.cos");
    for (int64_t k = 0; k < n; ++k) {
        if (op == 0) out[k] = lsm_sin(a[k]);
        else if (op == 1) out[k] = lsm_cos(a[k]);
        else if (op == 2) out[k] = lsm_atan2(a[k], b[k]);
        else { double s, c; lsm_sincos(a[k], &s, &c); out[k] = op == 3 ? s : c; }
    }
    return 0;
}

int lsm_math_eval_device(int op, const double* a, const double* b, double* out, int64_t n, void* stream) {
    if (a == nullptr || out == nullptr || (op == 2 && b == nullptr)) return fail(1, "lsm_math_eval_device: null argument");
    if (op < 0 || op > 4) return fail(2, "lsm_math_eval_device: bad op");
    cudaError_t e = lsm::math_eval_launch(op, a, b, out, (long long)n, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "lsm_math_eval_device");
    return 0;
}

int lsm_invalidate(lsm_handle* h) {
    if (h == nullptr) return fail(1, "lsm_invalidate: null handle");
    h->pairval_valid = false;
    return 0;
}

int lsm_emit_only(lsm_handle* h, void* stream) {
    if (h == nullptr) return fail(1, "lsm_emit_only: null handle");
    if (!h->have_buffers) return fail(5, "lsm_emit_only: lsm_bind_buffers has not been called");
    if (!h->spec) return fail(6, "lsm_emit_only: this configuration runs the fused generic kernel (no separate emission launch)");
    lsm::KParams kp = h->kp;
    kp.mode = lsm::MODE_OBSERVE; kp.env_mask = nullptr;
    DeviceGuard guard(h->device);
    kp.pair_late = 0;
    kp.grp_begin = 0; kp.env_begin = 0; kp.env_end = (int)kp.b.num_envs;
    if (kp.edge_index != nullptr && h->chunks > 1) kp.edge_index = nullptr;   // the per-range prefixes of a chunked step do not describe one launch
    kp.edge_range = 0; kp.edge_num_ranges = 1;
    kp.edge_envs_per_block = lsm::edge_count_envs_per_block(kp.b.num_envs); kp.edge_block_ofs = 0;
    kp.pairval = nullptr;     // the same kernel, grid and work as inside lsm_step
    cudaError_t e = lsm::spec_launch_emit(kp, h->tab, h->sm_count, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "lsm_emit_only");
    return 0;
}

int lsm_copy_records(lsm_handle* h, void* dst, void* stream) {
    if (h == nullptr) return fail(1, "lsm_copy_records: null handle");
    if (!h->spec) return fail(6, "lsm_copy_records: this configuration runs the fused generic kernel (no emit records)");
    if (!h->have_buffers) return fail(5, "lsm_copy_records: lsm_bind_buffers has not been called");
    if (dst == nullptr) return fail(2, "lsm_copy_records: null destination");
    DeviceGuard guard(h->device);
    const size_t bytes = (size_t)h->kp.b.num_envs * (size_t)h->tab.rec_bytes;
    const cudaError_t e = cudaMemcpyAsync(dst, h->d_emit_rec, bytes, cudaMemcpyDefault, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "lsm_copy_records");
    return 0;
}

int lsm_emit_from_records(lsm_handle* h, const lsm_record_emit_io* io, void* stream) {
    if (h == nullptr || io == nullptr) return fail(1, "lsm_emit_from_records: null argument");
    if (!h->spec) return fail(6, "lsm_emit_from_records: this configuration runs the fused generic kernel (no emit records)");
    if (io->num_items < 0 || io->num_records < 0) return fail(2, "lsm_emit_from_records: num_items and num_records must be >= 0");
    if (io->num_items == 0 || (io->node_obs == nullptr && io->adj == nullptr)) return 0;
    if (io->record == nullptr || io->observer == nullptr) return fail(2, "lsm_emit_from_records: record and observer are required");
    if (io->num_records > 0 && io->records == nullptr) return fail(2, "lsm_emit_from_records: null record store");
    if (((uintptr_t)io->records & 15u) || ((uintptr_t)io->node_obs & 15u) || ((uintptr_t)io->adj & 15u))
        return fail(2, "lsm_emit_from_records: records, node_obs and adj must be 16-byte aligned");
    DeviceGuard guard(h->device);
    lsm::RecordEmitArgs a;
    a.num_items = io->num_items; a.num_records = io->num_records;
    a.records = (const unsigned char*)io->records; a.record = (const long long*)io->record; a.observer = io->observer;
    a.node_obs = io->node_obs; a.adj = io->adj;
    a.sel_tab = h->kp.sel_tab; a.r2_lt = h->kp.r2_lt; a.r2_nz = h->kp.r2_nz;
    a.gfeat = (h->kp.c.flags & LSM_FLAG_GRAPH_FEAT_GLOBAL) != 0;
    const cudaError_t e = lsm::spec_launch_record_emit(h->tab, h->sm_count, a, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "lsm_emit_from_records");
    return 0;
}

int lsm_edges_from_records(lsm_handle* h, const lsm_record_edges_io* io, void* stream) {
    if (h == nullptr || io == nullptr) return fail(1, "lsm_edges_from_records: null argument");
    if (!h->spec) return fail(6, "lsm_edges_from_records: this configuration runs the fused generic kernel (no emit records)");
    if (io->num_items < 0 || io->num_records < 0 || io->capacity < 0)
        return fail(2, "lsm_edges_from_records: num_items, num_records and capacity must be >= 0");
    const bool fill = io->edge_index != nullptr;
    if (io->offsets == nullptr) return fail(2, "lsm_edges_from_records: offsets is required");
    if (io->num_items > 0) {
        if (fill ? io->edge_attr == nullptr : io->counts == nullptr)
            return fail(2, "lsm_edges_from_records: the count pass needs counts, the fill pass edge_attr");
        if (io->record == nullptr || io->observer == nullptr) return fail(2, "lsm_edges_from_records: record and observer are required");
        if (io->num_records > 0 && io->records == nullptr) return fail(2, "lsm_edges_from_records: null record store");
        if ((uintptr_t)io->records & 15u) return fail(2, "lsm_edges_from_records: records must be 16-byte aligned");
    }
    DeviceGuard guard(h->device);
    lsm::RecordEdgesArgs a;
    a.num_items = io->num_items; a.num_records = io->num_records;
    a.records = (const unsigned char*)io->records; a.record = (const long long*)io->record; a.observer = io->observer;
    a.counts = io->counts; a.offsets = (const long long*)io->offsets;
    a.edge_index = (long long*)io->edge_index; a.edge_attr = io->edge_attr; a.capacity = io->capacity;
    a.sel_tab = h->kp.sel_tab; a.r2_lt = h->kp.r2_lt; a.r2_nz = h->kp.r2_nz;
    const cudaError_t e = lsm::spec_launch_record_edges(h->tab, h->sm_count, a, (long long*)io->offsets, fill, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "lsm_edges_from_records");
    return 0;
}

int lsm_debug_pair_values(lsm_handle* h, double* out, void* stream) {
    if (h == nullptr) return fail(1, "lsm_debug_pair_values: null handle");
    if (!h->have_buffers) return fail(5, "lsm_debug_pair_values: lsm_bind_buffers has not been called");
    if (h->d_pairval == nullptr) return fail(6, "lsm_debug_pair_values: this configuration keeps no pair values");
    if (out == nullptr) return fail(2, "lsm_debug_pair_values: null output");
    DeviceGuard guard(h->device);
    const size_t bytes = (size_t)h->kp.b.num_envs * h->kp.N * h->kp.N * sizeof(double);
    const cudaError_t e = cudaMemcpyAsync(out, h->d_pairval, bytes, cudaMemcpyDefault, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "lsm_debug_pair_values");
    return 0;
}

// the standalone filter operator needs the handle's value grid only (no bound buffers)
static int filter_op_check_grid(const lsm_handle* h, const char* who) {
    if (!h->kp.has_vg) return fail(5, std::string(who) + ": the handle has no value grid (call lsm_set_value_grid first)");
    const int want = h->kp.c.dynamics == LSM_DYN_DOUBLE_INTEGRATOR ? 4 : 5;
    if (h->kp.vg.ndim != want) return fail(2, std::string(who) + ": the value grid's dimensionality does not match the dynamics");
    return 0;
}

int lsm_safety_filter(lsm_handle* h, const lsm_filter_io* io, void* stream) {
    if (h == nullptr || io == nullptr) return fail(1, "lsm_safety_filter: null argument");
    if (int rc = filter_op_check_grid(h, "lsm_safety_filter")) return rc;
    if (io->num_rows < 0 || io->num_slots < 0) return fail(2, "lsm_safety_filter: num_rows and num_slots must be >= 0");
    if (io->num_rows == 0) return 0;
    if (io->ego == nullptr || io->ego_action == nullptr || io->safe_action == nullptr)
        return fail(2, "lsm_safety_filter: ego, ego_action and safe_action are required");
    if (io->num_slots > 0 && (io->others == nullptr || io->other_actions == nullptr))
        return fail(2, "lsm_safety_filter: others and other_actions are required when num_slots > 0");
    DeviceGuard guard(h->device);
    lsm::FilterOpArgs a;
    a.rows = io->num_rows; a.slots = io->num_slots;
    a.ego = io->ego; a.others = io->others; a.ego_action = io->ego_action; a.other_actions = io->other_actions;
    a.active = io->active; a.sep = io->separation_distance;
    a.safe_action = io->safe_action; a.filtered = io->filtered; a.index = io->index; a.value = io->value;
    const cudaError_t e = lsm::safety_filter_launch(h->kp, h->sm_count, a, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "lsm_safety_filter");
    return 0;
}

int lsm_hj_lookup(lsm_handle* h, const lsm_lookup_io* io, void* stream) {
    if (h == nullptr || io == nullptr) return fail(1, "lsm_hj_lookup: null argument");
    if (int rc = filter_op_check_grid(h, "lsm_hj_lookup")) return rc;
    if (io->num_points < 0) return fail(2, "lsm_hj_lookup: num_points must be >= 0");
    if (io->num_points == 0) return 0;
    if (io->value == nullptr) return fail(2, "lsm_hj_lookup: value is required");
    if (io->rel == nullptr && (io->ego == nullptr || io->other == nullptr))
        return fail(2, "lsm_hj_lookup: give either rel or both ego and other");
    DeviceGuard guard(h->device);
    lsm::LookupArgs a;
    a.points = io->num_points; a.rel = io->rel; a.ego = io->ego; a.other = io->other; a.sep = io->separation_distance;
    a.value = io->value; a.grad = io->grad; a.rel_out = io->rel_out;
    const cudaError_t e = lsm::hj_lookup_launch(h->kp, h->sm_count, a, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "lsm_hj_lookup");
    return 0;
}

int lsm_debug_timeline(lsm_handle* h, int arm, uint64_t* out_ns) {
    if (h == nullptr) return fail(1, "lsm_debug_timeline: null handle");
    DeviceGuard guard(h->device);
    cudaError_t e;
    if (out_ns != nullptr && h->d_timeline != nullptr) {
        if ((e = cudaDeviceSynchronize()) != cudaSuccess) return cuda_fail(e, "lsm_debug_timeline");
        if ((e = cudaMemcpy(out_ns, h->d_timeline, sizeof(uint64_t) * lsm::TL_COUNT, cudaMemcpyDeviceToHost)) != cudaSuccess)
            return cuda_fail(e, "lsm_debug_timeline");
    }
    if (arm) {
        if (h->d_timeline == nullptr && (e = cudaMalloc(&h->d_timeline, sizeof(uint64_t) * lsm::TL_COUNT)) != cudaSuccess)
            return cuda_fail(e, "lsm_debug_timeline");
        uint64_t init[lsm::TL_COUNT];
        for (int k = 0; k < lsm::TL_COUNT; ++k) init[k] = 0;
        init[lsm::TL_PAIR_START] = init[lsm::TL_AGENT_START] = init[lsm::TL_EMIT_START] = ~0ull;
        if ((e = cudaMemcpy(h->d_timeline, init, sizeof(init), cudaMemcpyHostToDevice)) != cudaSuccess) return cuda_fail(e, "lsm_debug_timeline");
        h->kp.timeline = h->d_timeline;
    } else {
        h->kp.timeline = nullptr;
    }
    return 0;
}

}  // extern "C"

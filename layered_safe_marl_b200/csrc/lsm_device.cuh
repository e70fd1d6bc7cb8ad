// lsm_device.cuh - device-side building blocks of the fused step kernel (sm_100a).
//
// Arithmetic contract: every thresholded quantity (distances, HJ values, control differences,
// goal conditions) is computed in float64 in the reference's operation order and the translation
// unit is compiled with -fmad=false, so no product-sum is ever contracted into an FMA. Outputs are
// rounded to float32 only when they are stored.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/lsm_b200.h"
// float64 sin / cos / sincos / atan2 shared bit for bit with the CPU oracle (no libdevice / glibc rounding freedom)
#include "../../include/lsm_math.h"

namespace lsm {

constexpr double kPi = 3.141592653589793;
constexpr int kMaxAgents = LSM_MAX_AGENTS;
constexpr int kMaxLandmarks = LSM_MAX_LANDMARKS;
constexpr int kMagSegments = 50;

enum Mode { MODE_STEP = 0, MODE_RESET = 1, MODE_OBSERVE = 2 };

struct GridDev {
    int ndim;
    int shape[5];
    int periodic[5];
    double lo[5];
    double spacing[5];
    double inv_spacing[5];     // RN(1/spacing): exact division through the reciprocal (spec kernels)
    double separation_distance;
    double ttr_max;
    const float* values;
    const float* grads;
    // corner-packed copy of `values` (library-owned, built by lsm_set_value_grid): for every "lower corner" index tuple
    // the 2^ndim stencil values it anchors, contiguous in the corner order of the interpolation (binary counting, dim 0
    // slowest; upper index = lower + 1, wrapped on periodic dims, clamped at the last node otherwise). One lookup reads
    // one 64-byte (4-D) / 128-byte (5-D) aligned chunk instead of 2^ndim scattered words. NULL = not built.
    const float* packed;
    // 5-D grids: gradient rows padded from 5 to 8 floats (library-owned copy) so that one corner is two 16-byte loads
    // instead of five scalar ones. NULL = not built (4-D rows are one float4 already).
    const float* grads8;
    // LSM_FLAG_INTERP_FLOAT32: positions, weights and the corner sum in float32 (what jax computes without x64); 0 = float64
    int f32;
};

// per-env shared-memory block: element offsets (in bytes from the env block base)
struct SmemLayout {
    int ax, ay, as2, as3;                  // doubles [N]
    int vpre_x, vpre_y, vpost_x, vpost_y;  // doubles [N] world-frame velocity before / after own goal update
    int spd_post, sth, cth;                // doubles [N]
    int rawx, rawy;                        // doubles [N] decoded raw controls
    int lx, ly, lh, lsp, lsin, lcos;       // doubles [M]
    int ox, oy;                            // doubles [O] obstacle positions (obstacle extension)
    int daa;                               // doubles [N*N] agent-agent distances
    int dthr;                              // floats [E*E] radius-thresholded distances (16 B aligned)
    int goal_pre, goal_post, reached_pre, reached_post, done_pre, done_post;  // ints [N]
    int disc_pre, disc_post;               // uint32 [W]
    int keepm;                             // uint32 [N*W] per-observer keep masks
    int bytes_per_env;
};

struct KParams {
    lsm_config c;
    double sep_ratio_tab[5];   // 1 - cos(stair * pi/2) for stair = 0, 1/4, .., 1 (host libm)
    GridDev vg, tg;
    int has_vg, has_tg;
    lsm_buffers b;
    const int32_t* action_idx;
    const float* action_onehot;
    const uint8_t* env_mask;
    long long episode;
    unsigned long long seed;
    int mode;
    int flag;                  // STEP: auto_reset, RESET: sample
    int N, L, M, E, D, F;
    int O;                     // obstacles (declared extension, lsm_config.num_obstacles); E = N + M + O
    int G;                     // lanes per env (power of two >= N)
    int EPW;                   // envs per warp = 32 / G
    int W;                     // 32-bit mask words per entity set
    int adj_vec;               // 4, 2 or 1: widest aligned vector store usable for adj rows
    int smem_per_warp;
    SmemLayout sl;
    const uint16_t* pair_tab;  // [num_pairs][2] entity pairs a < b
    const uint32_t* pair32;    // [num_pairs] the same pairs packed (a << 16) | b
    int num_pairs;
    int ngroups;               // ceil(num_envs / EPW); with chunked launches: END of this launch's env-group range
    int grp_begin;             // first env group of this launch (chunked multi-stream launches; 0 otherwise)
    int env_begin, env_end;    // the same range in environments (emit / pair kernels)
    const uint32_t* sel_tab;   // [N][W] entities whose owner agent is <= i
    // exact squared thresholds (host): lt(T) = min{t : sqrt_rn(t) >= T} so that d < T <=> d2 < lt(T);
    //                                  gt(T) = min{t : sqrt_rn(t) >  T} so that d > T <=> d2 >= gt(T)
    double r2_lt, r2_gt;       // coordination_range (adjacency radius / filter range)
    double r2_nz;              // max{t : (float)sqrt_rn(t) == 0}: the float32 adjacency has an entry <=> r2_nz < d2 < r2_lt
    double col2_lt;            // 1.05 * (size + size) agent collision distance
    double engref2_lt;         // world.engagement_distance (episode statistics)
    double septgt2_lt;         // world.separation_distance_target (episode statistics)
    double sep2_lt[5], eng2_lt[5];   // scenario separation / engagement distance per curriculum stair level
    // specialised pipeline (library-owned scratch, L2 resident between the launches of one step)
    double* pairval;           // [num_envs][N][N] raw HJ value of (ego, other) from lsm_pair_kernel; NULL = compute in-kernel
    unsigned char* emit_rec;   // [num_envs][sizeof(EmitRec)] per-env record consumed by lsm_emit_kernel
    int pair_late;             // lsm_pair_kernel launched BEHIND the emit kernel of the same step (runs beside its drain)
    int pair_tail;             // the agent kernel itself computes the NEXT step's pair values at its tail (placement 4)
    int pair_rec;              // lsm_pair_kernel reads the emit records this launch's agent kernel wrote, not the SoA state
    float* adj_base;           // compact adjacency (lsm_set_compact_adjacency): [num_envs][E][E], NULL = dense adj output
    unsigned* adj_keep;        //                                             [num_envs][N][W]
    // fused COO edge output (lsm_set_edge_output, SURVEY 8f N2); edge_index == nullptr = off
    long long* edge_index;          // [2][edge_capacity]: row 0 = graph * E + row, row 1 = graph * E + col
    float* edge_attr;               // [edge_capacity]
    int* edge_counts;               // [num_envs * N] non-zeros per graph
    long long* edge_offsets;        // [num_envs * N + 1] global exclusive prefix, [graphs] = nnz
    long long edge_capacity;
    int* edge_local;                // library scratch [num_envs * N]: exclusive prefix inside the count block's env run
    long long* edge_block_totals;   // library scratch: edges of every count block / their exclusive prefix inside the range
    long long* edge_block_base;
    int edge_block_ofs;             // first entry of this launch's range in the two arrays above
    int edge_envs_per_block;        // environments per count block (contiguous run)
    long long* edge_range_totals;   // library scratch [16]: edges of every env range of the step
    unsigned* edge_tickets;         // library scratch [16]: block tickets of lsm_edge_count_kernel
    int edge_range, edge_num_ranges;
    int edge_dense;                 // 1: the dense adjacency is written as well
    unsigned long long* timeline;   // diagnostics (lsm_debug_timeline), NULL in production: globaltimer min-start / max-end per kernel
};

// lsm_emit_from_records: items (record, observer) of a caller-owned record store, re-emitted with a handle's constants
struct RecordEmitArgs {
    long long num_items, num_records;
    const unsigned char* records;   // [num_records][sizeof(EmitRec)], 16-byte aligned
    const long long* record;        // [num_items]
    const int* observer;            // [num_items]
    float* node_obs;                // [num_items][E][F or 7] or NULL
    float* adj;                     // [num_items][E][E] or NULL
    const uint32_t* sel_tab;        // KParams::sel_tab
    double r2_lt, r2_nz;            // KParams::r2_lt / r2_nz
    int gfeat;                      // LSM_FLAG_GRAPH_FEAT_GLOBAL
};

// lsm_edges_from_records: the COO edge list of the same items' matrices (count pass, then fill pass)
struct RecordEdgesArgs {
    long long num_items, num_records;
    const unsigned char* records;   // [num_records][sizeof(EmitRec)], 16-byte aligned
    const long long* record;        // [num_items]
    const int* observer;            // [num_items]
    int32_t* counts;                // count pass: [num_items] out
    const long long* offsets;       // fill pass: [num_items + 1], the count pass's prefix
    long long* edge_index;          // fill pass: [2][capacity]
    float* edge_attr;               // fill pass: [capacity]
    long long capacity;
    const uint32_t* sel_tab;        // KParams::sel_tab
    double r2_lt, r2_nz;            // KParams::r2_lt / r2_nz
};

// timeline slots: first block in / last block out of each kernel of the pipeline (ns, %globaltimer)
enum { TL_PAIR_START = 0, TL_PAIR_BODY_END, TL_AGENT_START, TL_AGENT_END, TL_EMIT_START, TL_EMIT_END, TL_PAIR_END, TL_COUNT };
__device__ __forceinline__ unsigned long long globaltimer_ns() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
__device__ __forceinline__ void tl_start(unsigned long long* tl, int slot) { if (tl != nullptr && threadIdx.x == 0) atomicMin(tl + slot, globaltimer_ns()); }
__device__ __forceinline__ void tl_end(unsigned long long* tl, int slot) { if (tl != nullptr && threadIdx.x == 0) atomicMax(tl + slot, globaltimer_ns()); }

__device__ __forceinline__ double clipd(double v, double lo, double hi) { return v < lo ? lo : (v > hi ? hi : v); }
__device__ __forceinline__ double pymax(double a, double b) { return (b > a) ? b : a; }
__device__ __forceinline__ double pymin(double a, double b) { return (b < a) ? b : a; }
__device__ __forceinline__ double norm2(double a, double b) { return sqrt(a * a + b * b); }
__device__ __forceinline__ double f32r(double v) { return (double)(float)v; }

// L2 eviction-priority hints (createpolicy): the 100 MB - 10 GB observation stream of one step is written evict-first
// and the HJ grids are gathered evict-last, so the stream does not push the few-MB grids out of the 126 MB L2 - without
// them the pair kernel's gathers miss to HBM and its reads interleave with the emit kernel's write stream.
__device__ __forceinline__ unsigned long long l2_evict_first() {
    unsigned long long p; asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p)); return p;
}
__device__ __forceinline__ unsigned long long l2_evict_last() {
    unsigned long long p; asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p)); return p;
}
__device__ __forceinline__ float ldg_hint(const float* p, unsigned long long pol) {
    float v; asm("ld.global.nc.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(v) : "l"(p), "l"(pol)); return v;
}
__device__ __forceinline__ float4 ldg_hint(const float4* p, unsigned long long pol) {
    float4 v;
    asm("ld.global.nc.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol));
    return v;
}

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011): counter based, keyed by (seed, env, reset_count), so a device
// reset can be replayed exactly by an independent CPU implementation of the same generator
// ---------------------------------------------------------------------------------------------
struct Rng {
    uint32_t k0, k1, env, reset_count, block;
    uint32_t buf[4];
    int have;
    __device__ void init(unsigned long long seed, uint32_t env_, uint32_t rc) {
        k0 = (uint32_t)seed; k1 = (uint32_t)(seed >> 32); env = env_; reset_count = rc; block = 0; have = 0;
    }
    __device__ void refill() {
        uint32_t c0 = block, c1 = env, c2 = reset_count, c3 = 0u, a = k0, b = k1;
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
            uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
            uint32_t n0 = hi1 ^ c1 ^ a, n1 = lo1, n2 = hi0 ^ c3 ^ b, n3 = lo0;
            c0 = n0; c1 = n1; c2 = n2; c3 = n3;
            a += 0x9E3779B9u; b += 0xBB67AE85u;
        }
        buf[0] = c0; buf[1] = c1; buf[2] = c2; buf[3] = c3;
        block++; have = 2;
    }
    __device__ double uniform01() {
        if (have == 0) refill();
        int k = 2 - have;
        have--;
        uint32_t a = (k == 0 ? buf[0] : buf[2]) >> 5, b = (k == 0 ? buf[1] : buf[3]) >> 6;
        return ((double)a * 67108864.0 + (double)b) / 9007199254740992.0;
    }
    __device__ double uniform(double lo, double hi) { return lo + (hi - lo) * uniform01(); }
};

// ---------------------------------------------------------------------------------------------
// Curriculum scalars: navigation_graph_safe.py:324-366, :1101-1122, :319-322
// ---------------------------------------------------------------------------------------------
struct Curriculum {
    double sloped, stair, heading_thresh, speed_thresh, dist_thresh;
    double multi_rew, conflict_rew, diff_rew, cvalue_rew, sep, eng;
    bool world_filter;
};

__device__ __forceinline__ double ratio_sloped(double ratio, double start, double end) {
    return clipd(ratio - start, 0.0, end - start) / (end - start);
}
__device__ __forceinline__ double ratio_stair(double ratio, int num_steps, double start, double end) {
    if (ratio < start) return 0.0;
    if (ratio > end) return 1.0;
    double cont = (double)(num_steps - 1) * clipd(ratio - start, 0.0, end - start) / (end - start);
    return (1.0 + floor(cont)) / (double)num_steps;
}
__device__ __forceinline__ Curriculum curriculum(const KParams& kp, double ratio) {
    const lsm_config& c = kp.c;
    Curriculum q;
    q.sloped = ratio_sloped(ratio, 0.25, 0.75);
    q.stair = ratio_stair(ratio, 4, 0.2, 0.75);
    q.heading_thresh = c.heading_thresh * (1.0 - q.sloped) + c.heading_thresh * q.sloped;
    q.speed_thresh = c.speed_thresh * (1.0 - q.stair) + c.speed_thresh * q.stair;
    q.dist_thresh = c.dist_thresh * (1.0 - q.stair) + c.dist_thresh * q.stair;
    q.multi_rew = c.potential_conflict_rew * q.stair;
    q.conflict_rew = c.safety_violation_rew * q.stair;
    q.diff_rew = c.diff_from_filtered_action_rew * q.stair;
    q.cvalue_rew = c.hj_value_rew * q.stair;
    // 1 - cos(stair * pi / 2): stair takes the five values k/4, the host tabulates them with libm
    const int k = (int)(q.stair * 4.0);
    const double sep_ratio = kp.sep_ratio_tab[k];
    const bool use_filter_arg = (c.flags & LSM_FLAG_USE_SAFETY_FILTER) != 0;
    const bool initial_phase = use_filter_arg && (c.flags & LSM_FLAG_INITIAL_PHASE_USE_SAFETY_FILTER);
    q.world_filter = use_filter_arg;
    if (!initial_phase && use_filter_arg) q.world_filter = q.sloped > 0.0;
    const double sep_init = (c.flags & LSM_FLAG_SEPARATION_DISTANCE_CURRICULUM) ? 0.0 : c.separation_distance_target;
    q.sep = sep_init * (1.0 - sep_ratio) + c.separation_distance_target * sep_ratio;
    q.eng = c.engagement_distance_ref + (q.sep - c.engagement_ref_separation);
    return q;
}

// utils.py:79-81
__device__ __forceinline__ double direction_alignment_error(double h, double href) { return 0.5 - 0.5 * lsm_cos(h - href); }

// utils.py:104-112 with precomputed cos / sin of the reference heading
__device__ __forceinline__ void rotate_into(double dx, double dy, double c, double s, double& ox, double& oy) {
    ox = c * dx + s * dy;
    oy = (-s) * dx + c * dy;
}

template <int DYN>
__device__ __forceinline__ double theta_of(double s2, double s3) { return DYN == LSM_DYN_DOUBLE_INTEGRATOR ? lsm_atan2(s3, s2) : s2; }
template <int DYN>
__device__ __forceinline__ double speed_of(double s2, double s3) {
    return DYN == LSM_DYN_DOUBLE_INTEGRATOR ? sqrt(s2 * s2 + s3 * s3) : s3;
}

// navigation_graph_safe.py:606-656
// `he` = direction_alignment_error(theta, goal heading), computed once by the caller (the reward needs it too)
template <int DYN>
__device__ __forceinline__ bool goal_reached_he(double x, double y, double he, double speed, double gx, double gy,
                                                double gs, const Curriculum& q) {
    const double dx = x - gx, dy = y - gy;
    const double dist = sqrt(dx * dx + dy * dy);
    const double ve = fabs(speed - gs);
    bool cond;
    if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) {
        const double speed_advantage_thresh = 0.2;
        if (dist > q.dist_thresh) cond = he < q.heading_thresh;
        else if (gs > speed_advantage_thresh) cond = he < q.heading_thresh;
        else {
            const double sa = clipd(1.0 - gs / speed_advantage_thresh, 0.0, 1.0);
            const double tc = 0.5 * sa + q.heading_thresh * (1.0 - sa);
            const double da = clipd(1.0 - dist / q.dist_thresh, 0.0, 1.0);
            const double tca = tc * da + q.heading_thresh * (1.0 - da);
            cond = he < tca;
        }
    } else cond = he < q.heading_thresh;
    return dist < q.dist_thresh && cond && ve < q.speed_thresh;
}
template <int DYN>
__device__ __forceinline__ bool goal_reached(double x, double y, double theta, double speed, double gx, double gy,
                                             double gh, double gs, const Curriculum& q) {
    return goal_reached_he<DYN>(x, y, direction_alignment_error(theta, gh), speed, gx, gy, gs, q);
}

// single-constraint QP (declared semantics; replaces cvxpy/OSQP at safety_filter.py:286-308,364-376)
__device__ __forceinline__ bool qp_project(const double (&a)[4], double b, const double (&r)[4],
                                           const double (&pinv)[4], double (&u)[4]) {
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < 4; ++k) s = s + a[k] * r[k];
    s = s + b;
    if (s >= 0.0) {
#pragma unroll
        for (int k = 0; k < 4; ++k) u[k] = r[k];
        return true;
    }
    double denom = 0.0;
#pragma unroll
    for (int k = 0; k < 4; ++k) denom = denom + (a[k] * pinv[k]) * a[k];
    if (denom == 0.0) return false;
    const double lam = s / denom;
#pragma unroll
    for (int k = 0; k < 4; ++k) u[k] = r[k] - lam * (pinv[k] * a[k]);
    return true;
}

}  // namespace lsm

// lsm_kernel_spec.cuh - the step pipeline specialised at compile time on (dynamics, N agents, L landmarks
// per agent): constant-size records, unrolled loops, immediate-offset stores.
//
// One env.step is THREE launches, each at the natural parallelism of its phase (a fused single kernel needs ~250
// registers for the physics and then runs the store-bound graph emission at 7 warps per SM; measured in
// profiles/r01_v3_*: 17 % issue utilisation, latency-bound), in stream order
//
//   lsm_agent_kernel  one LANE per agent, 32/N envs per warp: action decode, argmin over the precomputed HJ pair values /
//                     gradient / bang-bang or QP, dynamics, goal / reward / done, episode statistics, auto-reset, state
//                     write-back; leaves a compact per-env "emit record" (positions, velocities, goal tables, pre/post flags)
//   lsm_emit_kernel   persistent blocks of WPE warps loop over envs, low register count: radius-thresholded distance
//                     matrix, disconnected-entity masks, adjacency and node-feature tiles in shared memory -> TMA bulk
//                     stores - the HBM-bound part (>= 96 % of the algorithmic bytes)
//   lsm_pair_kernel   one THREAD per ordered (env, ego, other) pair: relative state + multilinear HJ value lookup from the
//                     corner-packed table (safety_filter.py:192-201, 345-354) -> pairval[env][ego][other] for the NEXT step;
//                     launched behind the emit kernel without a dependency wait, so it runs beside the emit kernel's drain
//
// Big batches are split into env ranges on library-owned streams (lsm_capi.cu) so that the latency-bound agent kernel of
// one range overlaps the HBM-bound emit kernel of another.
//
// Same decisions as the generic kernel for every thresholded quantity:
//   * the HJ grid lookups are the shared ones of lsm_grid.cuh (the value from the corner-packed table, which
//     reproduces the stencil bit for bit).
//   * distances are kept SQUARED in float64; every `d < T` / `d > T` test of the reference becomes
//     `d2 < T2` against a host-computed exact squared threshold (sqrt_rn is monotone, so
//     {t : sqrt_rn(t) >= T} is an interval whose lower end the host finds with nextafter). Square roots
//     are taken only where a distance VALUE is stored (min distance, float32 adjacency).
//   * the float32 adjacency value is d2f * rsqrt(d2f) (<= 4e-7 relative from the float64 reference, bar
//     1e-5; a distance below 1e-15 is stored as 1e-15); which entries are non-zero is decided exactly in float64,
//     strictly inside the radius and above the largest d2 whose float32 root is 0 (r2_nz).
//   * node features are branch-free rows over unified per-entity tables (landmarks carry zero velocity and
//     their own position as "goal"), read with 16-byte shared-memory loads.
#pragma once
#include "lsm_step_common.cuh"

namespace lsm {

// airtaxi-only part of the emit record (rotations into the observer frame need float64 sin / cos)
template <int DYN, int N, int L, int O>
struct AirExtra {
    double sth[N], cth[N], spd_post[N];           // sin/cos(theta), speed after the own update
    double theta[N];                              // heading (never changed by the goal update)
    double lsin[N * L + O], lcos[N * L + O], lsp[N * L + O];   // landmark sin/cos(heading), speed; obstacles: (0, 1, 0)
    int goal[2][N];                                // landmark index of the goal before / after the own update
};
template <int N, int L, int O>
struct AirExtra<LSM_DYN_DOUBLE_INTEGRATOR, N, L, O> {};

// What the graph emission needs from the physics of one environment (written by lsm_agent_kernel, read by
// lsm_emit_kernel). Unified per-entity tables for the branch-free node-feature rows:
//   pos[e]                     position of entity e (agents after the dynamics, then landmarks)
//   pos[E + s*N + a]           goal position of agent a before (s=0) / after (s=1) its own goal update
//   vel[s*N + a], vel[2N] = 0  world-frame velocity of agent a before / after its update; landmarks use slot 2N
//   cst[m], cst[CA + s*N + a]  (sin heading, cos heading, speed, type) of landmark m / of agent a's goal
// O > 0 (declared obstacle extension, lsm_b200.h num_obstacles): obstacle k is entity N + M + k - pos[N + M + k], and
// cst[M + k] = (0, 1, 0, 2): the landmark row with heading 0, speed 0 and entity type 2; CA = M + O.
template <int DYN, int N, int L, int O>
struct __align__(16) EmitRec {
    static constexpr int M = N * L;
    static constexpr int E = N + M + O;
    static constexpr int W = (E + 31) / 32;
    static constexpr int CA = M + O;      // first agent-goal entry of cst
    // the domain lsm_create accepts (lsm_b200.h LSM_MAX_*): 8-bit landmark indices, 16-bit entity indices in pair_tab
    static_assert(N >= 1 && N <= LSM_MAX_AGENTS, "1 <= N <= 32: one lane per agent");
    static_assert(L >= 2 && M <= LSM_MAX_LANDMARKS, "L >= 2 and N * L <= 128");
    static_assert(O >= 0 && O <= LSM_MAX_OBSTACLES, "0 <= O <= 32");
    static_assert(W <= 6, "at most 192 entities: 6 mask words");
    double2 pos[E + 2 * N];
    double2 vel[2 * N + 1];
    float4 cst[M + O + 2 * N];
    int reached[2][N], done[2][N];
    int next_filter;           // world.use_safety_filter this env will have at the NEXT step (curriculum after a reset)
    int _pad[3];
    AirExtra<DYN, N, L, O> air;
};

// physics-only shared-memory scratch of one environment inside lsm_agent_kernel
template <int DYN, int N, int L>
struct __align__(16) AgentScratch {
    static constexpr int M = N * L;
    double as2[N], as3[N];     // state components 2,3 BEFORE the own goal update (vx,vy | theta,speed)
    double rawx[N], rawy[N];   // decoded raw controls
    double lh[M], lsp[M], lsin[M], lcos[M];   // landmark heading, speed, sin/cos(heading)
    double fval[N * N];        // HJ value of (ego i, other j) when computed in-kernel (internal steps > 1)
    double cur_sep;            // scenario.separation_distance of this env (curriculum)
    int cur_filter;            // world.use_safety_filter of this env (curriculum, Q5)
    int _pad;
};

// Programmatic dependent launch (griddepcontrol): every kernel of the pipeline is launched with
// cudaLaunchAttributeProgrammaticStreamSerialization, lets its successor become resident early (launch_dependents at
// the top) and waits for the complete, flushed predecessor before it touches global memory (wait). This hides the
// launch + block-dispatch latency (~6 us per launch in the bench's event timing) behind the predecessor's tail.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// fire-and-forget L2 prefetch: the per-agent kernel is a latency chain, and every input it touches late (pair values,
// actions, landmark tables, the parity-selected info slots) would otherwise be one more dependent DRAM round trip
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" :: "l"(p)); }

template <int N> struct Pow2 { static constexpr int value = N <= 1 ? 1 : N <= 2 ? 2 : N <= 4 ? 4 : N <= 8 ? 8 : N <= 16 ? 16 : 32; };

// raw (unshifted) HJ value of the pair (ego, other); +inf = outside the declared range / NaN
template <int DYN, bool F32 = false>
__device__ __forceinline__ double pair_value_raw(const GridDev& vg, double ex, double ey, double e2, double e3,
                                                 double ox, double oy, double o2, double o3) {
    // safety_filter.py:192-201, 345-354
    constexpr int ND = DYN == LSM_DYN_DOUBLE_INTEGRATOR ? 4 : 5;
    double rel[ND];
    relative_state_rot<DYN>(ex, ey, e2, e3, ox, oy, o2, o3, rel);
    return pair_value_rel<ND, kPeriodicRuntime, F32>(vg, rel);
}

// Relative state of (ego i, other j) from an emit record, i.e. from the state the agent kernel left behind: positions
// after the dynamics, velocity (double integrator) / heading and speed (airtaxi) after the own goal update - exactly
// the state it writes back to the SoA tensors. The airtaxi ego frame uses the record's (sth, cth): every path that
// writes a record takes them from lsm_sincos(theta) of the heading the record carries (integrate() after the
// dynamics, the observe / reset branches), the same function relative_state_rot evaluates per pair.
template <int DYN, int N, int L, int O>
__device__ __forceinline__ void pair_rel_rec(const EmitRec<DYN, N, L, O>& R, int i, int j,
                                             double (&rel)[DYN == LSM_DYN_DOUBLE_INTEGRATOR ? 4 : 5]) {
    const double2 pi = R.pos[i], pj = R.pos[j];
    if constexpr (DYN == LSM_DYN_DOUBLE_INTEGRATOR) {
        const double2 vi = R.vel[N + i], vj = R.vel[N + j];
        relative_state_rot_sc<DYN>(pi.x, pi.y, vi.x, vi.y, pj.x, pj.y, vj.x, vj.y, 0.0, 1.0, rel);
    } else {
        relative_state_rot_sc<DYN>(pi.x, pi.y, R.air.theta[i], R.air.spd_post[i], pj.x, pj.y, R.air.theta[j],
                                   R.air.spd_post[j], R.air.sth[i], R.air.cth[i], rel);
    }
}

// value shift of HjDataHandle.update_separation_distance (safety_filter.py:170-174); inf stays inf
__device__ __forceinline__ double shift_value(double raw, double sep, const GridDev& vg) {
    return raw - (sep - vg.separation_distance);
}

// ---------------------------------------------------------------------------------------------
// K_a: HJ values of every ordered agent pair, one thread per (env, ego, other).
//
// The values feed the NEXT step's filter (safety_filter.py:192-201 evaluates V(x_i - x_j) at the start of a step) and
// depend only on the state the agent kernel of THIS step left behind. Normal placement ("late"): launched right behind
// the emit kernel with programmatic dependent launch and WITHOUT a grid-dependency wait at its top - the emit kernel
// releases its dependents only after its own wait, i.e. once the agent kernel is complete and flushed - so these
// latency-bound L2 gathers run on the issue slots the store-bound emit kernel leaves idle, at full thread-per-pair
// parallelism. Block 0 waits for the emit kernel before it retires, which keeps "this grid complete" => "emit grid
// complete" for the next step's agent kernel. Middle placement (pair_late == 0): between the agent and the emit kernel.
// Fallback placement: in front of the agent kernel, when the state was edited from outside (lsm_invalidate / set_state).
//
// One thread per ORDERED pair i != j: N(N-1) tasks per env (r -> i = r / (N-1), j = r % (N-1) skipping i), 32-bit task
// indices (spec_launch_pair bounds the range), divisors known at compile time. pairval keeps its [env][N][N] layout;
// the diagonal is never written or read.
//
// Where the inputs come from (kp.pair_rec, chosen per launch in lsm_capi.cu):
//   * pair_rec = 1: the emit record this launch's agent kernel wrote for the env (pair_rel_rec): positions, velocity /
//     heading + speed, the done flags after the step and next_filter (the curriculum decision for the state the record
//     describes). Behind the agent kernel the record describes exactly the state it wrote back to the SoA tensors, in
//     every launch that writes the record of every env of the range: step (with or without auto-reset; the reset
//     branch rewrites the record), unmasked reset (sampled, or reset_from_state), observe.
//   * pair_rec = 0: the SoA state tensors and the curriculum ratio. In front of the agent kernel (the state may have
//     been edited after the last record was written), and behind a masked reset, which leaves the records of envs
//     outside the mask untouched (they may predate a set_state or never have been written).
//
// F32 = LSM_FLAG_INTERP_FLOAT32: the float32 lookup from the same corner-packed table (packed_value<.., true>).
// ---------------------------------------------------------------------------------------------
constexpr int kPairThreads = 128;
template <int DYN, int N, int L, int O, int PER, bool F32>
__global__ void __launch_bounds__(kPairThreads) lsm_pair_kernel(const __grid_constant__ KParams kp) {
    using REC = EmitRec<DYN, N, L, O>;
    constexpr int ND = DYN == LSM_DYN_DOUBLE_INTEGRATOR ? 4 : 5;
    constexpr unsigned T = N * (N - 1);
    constexpr unsigned TD = T > 0 ? T : 1, ND1 = N > 1 ? N - 1 : 1;   // N = 1: no tasks; the divisors stay non-zero
    pdl_launch_dependents();
    if (!kp.pair_late) pdl_wait();
    tl_start(kp.timeline, TL_PAIR_START);
    const unsigned tasks = (unsigned)(kp.env_end - kp.env_begin) * T;
    // grid-stride: the late placement runs a bounded number of blocks per SM (lsm_kernels.cu) so that these fp64-heavy
    // warps take a fixed share of the issue slots next to the emit kernel's producers
    for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < tasks; t += gridDim.x * blockDim.x) {
        const unsigned el = t / TD, r = t - el * TD;
        const int i = (int)(r / ND1), jj = (int)(r - (unsigned)i * ND1);
        const int j = jj + (jj >= i);
        const int env = kp.env_begin + (int)el;
        double rel[ND];
        if (kp.pair_rec) {
            const REC& R = reinterpret_cast<const REC*>(kp.emit_rec)[env];
            if (!R.next_filter || R.done[1][i] || R.done[1][j]) continue;
            pair_rel_rec<DYN, N, L, O>(R, i, j, rel);
        } else {
            const size_t n = (size_t)kp.b.num_envs;
            // world.use_safety_filter of this env (curriculum, navigation_graph_safe.py:351-357)
            if (!(kp.c.flags & LSM_FLAG_INITIAL_PHASE_USE_SAFETY_FILTER)) {
                const double ratio = kp.b.env_f64[(size_t)LSM_EF_CURRICULUM_RATIO * n + env];
                if (!(ratio_sloped(ratio, 0.25, 0.75) > 0.0)) continue;
            }
            const size_t fs = n * N;
            const size_t ia = (size_t)env * N + i, ja = (size_t)env * N + j;
            const int* dn = kp.b.agent_i32 + LSM_AI_DONE * fs;
            if (dn[ia] || dn[ja]) continue;
            const double* af = kp.b.agent_f64;
            relative_state_rot<DYN>(af[LSM_AF_X * fs + ia], af[LSM_AF_Y * fs + ia], af[LSM_AF_S2 * fs + ia],
                                    af[LSM_AF_S3 * fs + ia], af[LSM_AF_X * fs + ja], af[LSM_AF_Y * fs + ja],
                                    af[LSM_AF_S2 * fs + ja], af[LSM_AF_S3 * fs + ja], rel);
        }
        kp.pairval[(size_t)env * (N * N) + (i * N + j)] = pair_value_rel<ND, PER, F32>(kp.vg, rel);
    }
    tl_end(kp.timeline, TL_PAIR_BODY_END);
    if (kp.pair_late && blockIdx.x == 0 && threadIdx.x == 0) pdl_wait();
    tl_end(kp.timeline, TL_PAIR_END);
}

// in-kernel variant for internal steps after the first (states changed inside the launch): pair-parallel over
// the warp's environments, shifted values into P.fval
template <int DYN, int N, int L, int O, bool F32>
__device__ __noinline__ void pair_phase(const GridDev* __restrict__ vg, EmitRec<DYN, N, L, O>* Rw, AgentScratch<DYN, N, L>* Pw,
                                       int nenv, int lane) {
    const GridDev& g = *vg;
    for (int t = lane; t < nenv * N * N; t += 32) {
        const int el = t / (N * N), r = t - el * (N * N);
        const int i = r / N, j = r - i * N;
        const EmitRec<DYN, N, L, O>& R = Rw[el];
        AgentScratch<DYN, N, L>& P = Pw[el];
        if (!P.cur_filter || i == j || R.done[0][i] || R.done[0][j]) continue;
        const double2 pi = R.pos[i], pj = R.pos[j];
        P.fval[r] = shift_value(pair_value_raw<DYN, F32>(g, pi.x, pi.y, P.as2[i], P.as3[i], pj.x, pj.y, P.as2[j], P.as3[j]),
                                P.cur_sep, g);
    }
}

// placement 4 ("tail"): the agent kernel computes the NEXT step's pair values itself, right after it has left the state
// and the emit records behind (safety_filter.py:192-201 evaluates V(x_i - x_j) at the start of a step, from exactly this
// state). The per-agent chain is latency bound (~20 % issue utilisation), so these lookups ride on idle issue slots of
// warps that are resident anyway - no pair kernel competing with the emit kernel for the SMs, one launch less. Same
// conditions and arithmetic as lsm_pair_kernel (raw values; entries of done agents / filter-off envs are left alone).
template <int DYN, int N, int L, int O, bool F32>
__device__ __noinline__ void pair_tail_phase(const GridDev* __restrict__ vg, const EmitRec<DYN, N, L, O>* Rw, double* __restrict__ pairval,
                                            int env0, int nenv, unsigned on_mask, int lane) {
    const GridDev& g = *vg;
    for (int t = lane; t < nenv * N * N; t += 32) {
        const int el = t / (N * N), r = t - el * (N * N);
        const int i = r / N, j = r - i * N;
        const EmitRec<DYN, N, L, O>& R = Rw[el];
        if (!((on_mask >> ((el * N) & 31)) & 1u) || !R.next_filter || i == j || R.done[1][i] || R.done[1][j]) continue;
        double rel[DYN == LSM_DYN_DOUBLE_INTEGRATOR ? 4 : 5];
        pair_rel_rec<DYN, N, L, O>(R, i, j, rel);
        pairval[(size_t)(env0 + el) * (N * N) + r] = pair_value_rel<DYN == LSM_DYN_DOUBLE_INTEGRATOR ? 4 : 5, kPeriodicRuntime, F32>(g, rel);
    }
}

template <int DYN, int N, int L, int O>
__device__ __forceinline__ void emit_obs_row(const EmitRec<DYN, N, L, O>& R, const AgentScratch<DYN, N, L>& P, int ai,
                                             int g /* landmark index */, double x, double y, double s2, double s3, float* o) {
    // navigation_graph_safe.py:855-875, utils.py:114-137
    const double2 gp = R.pos[N + g];
    if constexpr (DYN == LSM_DYN_DOUBLE_INTEGRATOR) {
        o[0] = (float)s2; o[1] = (float)s3; o[2] = (float)(gp.x - x); o[3] = (float)(gp.y - y);
        o[4] = (float)P.lsin[g]; o[5] = (float)P.lcos[g]; o[6] = (float)P.lsp[g];
    } else {
        double rx, ry; rotate_into(gp.x - x, gp.y - y, R.air.cth[ai], R.air.sth[ai], rx, ry);
        // sin / cos(goal heading - theta) by the angle-difference identity over the tabulated landmark and own sin / cos
        // (<= 1e-15 from the reference expression, like the node features)
        const double ci = R.air.cth[ai], si = R.air.sth[ai];
        o[0] = (float)s3; o[1] = (float)rx; o[2] = (float)ry;
        o[3] = (float)(P.lsin[g] * ci - P.lcos[g] * si); o[4] = (float)(P.lcos[g] * ci + P.lsin[g] * si); o[5] = (float)P.lsp[g];
    }
}

// ---------------------------------------------------------------------------------------------
// TMA bulk store (UBLKCP): shared -> global, asynchronous, issued by one lane; frees the warp from
// the store loop and its LSU back-pressure. Source and destination 16-byte aligned, size % 16 == 0.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void bulk_store_fence() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void bulk_store(void* gdst, const void* ssrc, unsigned bytes) {
    const unsigned saddr = (unsigned)__cvta_generic_to_shared(ssrc);
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" :: "l"(gdst), "r"(saddr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_store(void* gdst, const void* ssrc, unsigned bytes, unsigned long long pol) {
    const unsigned saddr = (unsigned)__cvta_generic_to_shared(ssrc);
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
                 :: "l"(gdst), "r"(saddr), "r"(bytes), "l"(pol) : "memory");
}
__device__ __forceinline__ void bulk_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int PENDING>
__device__ __forceinline__ void bulk_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" :: "n"(PENDING) : "memory"); }

// Scenario.random_scenario for ONE environment, executed by the env's leader lane
// (navigation_graph_safe.py:1199-1367, utils.py:39-68); Philox stream keyed by (seed, env, reset_count).
template <int DYN, int N, int L, int O>
__device__ __noinline__ void sample_scenario(const KParams& kp, EmitRec<DYN, N, L, O>& R, AgentScratch<DYN, N, L>& P,
                                            int env, int reset_count, double ratio) {
    constexpr int M = N * L;
    const lsm_config& c = kp.c;
    const bool use_filter_arg = (c.flags & LSM_FLAG_USE_SAFETY_FILTER) != 0;
    Rng r; r.init(kp.seed, (uint32_t)(kp.b.env_id_base + env), (uint32_t)reset_count);
    const double ws = c.world_size;
    double cra = ratio_sloped(ratio, 0.25, 0.75);
    if (use_filter_arg) cra = 1.0;
    // static obstacles first (:1204-1209): 0.8 * uniform(-ws/2, ws/2, 2)
    for (int k = 0; k < O; ++k) {
        const double ox = 0.8 * r.uniform(-ws / 2.0, ws / 2.0);
        const double oy = 0.8 * r.uniform(-ws / 2.0, ws / 2.0);
        R.pos[N + M + k] = make_double2(ox, oy);
    }
    for (int i = 0; i < N; ++i) {
        // :1218-1249: with obstacles the position is redrawn while it collides with one (bounded at 1000 tries); the
        // airtaxi speed / heading are drawn once the position is accepted
        double px = 0.0, py = 0.0;
        for (int tries = 0; tries < (O > 0 ? 1000 : 1); ++tries) {
            if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) {
                px = r.uniform(-0.8 * ws, 0.8 * ws);
                py = r.uniform(-0.8 * ws, 0.8 * ws);
            } else {
                const double xmin = -0.5 * ws;
                const double xmax = 0.25 * ws * cra + 0.0 * (1.0 - cra) * ws;
                py = r.uniform(-0.5 * ws, 0.5 * ws);
                px = r.uniform(xmin, xmax);
            }
            bool hit = false;
            for (int k = 0; k < O; ++k) {      // navigation_graph_safe.py:452-465
                const double2 po = R.pos[N + M + k];
                const double dx = po.x - px, dy = po.y - py;
                if (dx * dx + dy * dy < kp.col2_lt) { hit = true; break; }
            }
            if (!hit) break;
        }
        R.pos[i] = make_double2(px, py);
        if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) { P.as2[i] = 0.0; P.as3[i] = 0.0; }
        else {
            const double sp = r.uniform(c.goal_speed_min, c.goal_speed_max);
            P.as2[i] = r.uniform(0.0, 2.0 * kPi);
            P.as3[i] = sp;
        }
    }
    double2* lp = R.pos + N;    // landmark positions, slot l*N + i
    for (int i = 0; i < N; ++i) {
        double xlo, xhi, ylo, yhi, min_d, max_d;
        if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) {
            xlo = -0.5 * ws; xhi = 0.5 * ws; ylo = -0.5 * ws; yhi = 0.5 * ws;
            min_d = 0.25 * c.coordination_range; max_d = 0.75 * c.coordination_range;
        } else {
            const double yw = 0.1 * (1.0 - cra) + 0.5 * cra;
            xlo = 0.0; xhi = 0.75 * ws; ylo = -yw * ws; yhi = yw * ws;
            min_d = 0.5 * c.coordination_range; max_d = c.coordination_range;
        }
        for (int l = 0; l < L; ++l) {
            double gx = 0.0, gy = 0.0;
            if (l > 0) {
                for (int j = 0; j < 1000; ++j) {
                    gx = r.uniform(xlo, xhi); gy = r.uniform(ylo, yhi);
                    double dm = INFINITY;
                    for (int k = 0; k < l; ++k) {
                        const double d = norm2(lp[k * N + i].x - gx, lp[k * N + i].y - gy);
                        if (d < dm) dm = d;
                    }
                    if (dm > min_d && dm < max_d) break;
                }
            } else { gx = r.uniform(xlo, xhi); gy = r.uniform(ylo, yhi); }
            lp[l * N + i] = make_double2(gx, gy);
        }
        if (i > 0) for (int l = 0; l < L; ++l) if (r.uniform(0.0, 1.0) < 0.5) lp[l * N + i] = lp[l * N + i - 1];
        if (DYN != LSM_DYN_DOUBLE_INTEGRATOR) {
            if (lp[i].x > lp[N + i].x) { const double2 t = lp[i]; lp[i] = lp[N + i]; lp[N + i] = t; }
        }
        for (int l = 0; l < L - 1; ++l)
            P.lh[l * N + i] = lsm_atan2(lp[(l + 1) * N + i].y - lp[l * N + i].y, lp[(l + 1) * N + i].x - lp[l * N + i].x);
        const double last_heading = P.lh[(L - 2) * N + i];
        const double cr = use_filter_arg ? 1.0 : ratio_sloped(ratio, 0.25, 0.75);
        if (DYN != LSM_DYN_DOUBLE_INTEGRATOR) {
            for (int l = 0; l < L; ++l) P.lsp[l * N + i] = c.goal_speed_max;
        } else {
            for (int l = 0; l < L; ++l) P.lsp[l * N + i] = r.uniform(c.goal_speed_min, c.goal_speed_max);
            const double var = r.uniform(0.0, 1.0);
            if (!(var < pymin(cr, 1.0 - 0.2))) {
                for (int l = 0; l < L; ++l) P.lsp[l * N + i] = c.goal_speed_max;
                P.lsp[(L - 1) * N + i] = c.goal_speed_min;
            }
        }
        for (int l = 0; l < L - 1; ++l) {
            const double pr = (DYN == LSM_DYN_DOUBLE_INTEGRATOR) ? cr * 0.25 * kPi : cra * 0.1 * kPi;
            P.lh[l * N + i] += r.uniform(-pr, pr);
        }
        P.lh[(L - 1) * N + i] = last_heading;
    }
    for (int m = 0; m < M; ++m) {
        double sv, cv;
        lsm_sincos_inl(P.lh[m], &sv, &cv);     // the out-of-line lsm_sincos would put sv / cv in local memory
        P.lsin[m] = sv; P.lcos[m] = cv;
        R.cst[m] = make_float4((float)sv, (float)cv, (float)P.lsp[m], 1.0f);
    }
}
// ---------------------------------------------------------------------------------------------
// Cold paths of the per-agent kernel, kept OUT OF LINE: the kernel runs its straight-line code once per
// warp, so its cost is dominated by instruction fetch (profiles/r01_v4b: stall_no_instruction 5.8 per
// issue); every rarely-taken block that is inlined becomes a far jump over kilobytes of SASS.
// ---------------------------------------------------------------------------------------------
// utils.py:323-349 (double integrator without the safety-filter argument): heading/velocity penalty
__device__ __noinline__ double magnetic_penalty(double x, double y, double s2, double s3, double gx, double gy,
                                               double gh, double gs, double dist_thresh, double sloped) {
    const double cg = lsm_cos(gh), sg = lsm_sin(gh);
    double rpx, rpy, rvx, rvy;
    rotate_into(x - gx, y - gy, cg, sg, rpx, rpy);
    const double dist = norm2(rpx, rpy);
    const double ang = lsm_atan2(rpy, rpx);
    const double ang_range = kPi / 6;
    rotate_into(s2 - 0.0, s3 - 0.0, cg, sg, rvx, rvy);
    const double rh = magnetic_heading(rpx, rpy, 2.0 * dist_thresh);
    double ref_speed = pymax(gs, 0.1);
    const double dr = clipd(dist / 1.5, 0.0, 1.0);
    ref_speed = ref_speed * (1.0 - dr) + 1.0 * dr;
    const double ex = rvx - ref_speed * lsm_cos(rh), ey = rvy - ref_speed * lsm_sin(rh);
    const double err = norm2(ex, ey);
    double pen;
    if (lsm_cos(ang) < lsm_cos(ang_range)) pen = err;
    else {
        const double ar = clipd((lsm_cos(ang) - lsm_cos(ang_range)) / (1.0 - lsm_cos(ang_range)), 0.0, 1.0);
        pen = err * (1.0 - ar) + dist * ar;
    }
    double hap = 3.0 * pen;
    hap = clipd(1.0 - sloped, 0.0, 1.0) * hap;
    return hap;
}

// navigation_graph_safe.py:700-720: heading * speed * cross-track factor of the goal reward (only on the step a goal is
// reached); (sth, cth) = lsm_sincos(theta)
__device__ __forceinline__ double goal_reward_factor(double sth, double cth, double pdx, double pdy, double hpr, double sen) {
    const double spr = 1.0 - sen;
    double cte = pdx * sth - pdy * cth;
    const double nrm = norm2(pdx, pdy);
    cte = fabs(cte) / (nrm > 1e-6 ? nrm : 1e-6);
    cte = clipd(cte, 0.0, 1.0);
    return hpr * spr * (1.0 - cte);
}

// reward_multiple_engagement (navigation_graph_safe.py:800-823) over the agents flagged in `mask`
template <int DYN, int N, int L, int O>
__device__ __noinline__ double potential_conflict_penalty(const EmitRec<DYN, N, L, O>& R, unsigned mask, int ai, double x, double y,
                                                         double vpx, double vpy, double sep, double eng) {
    double pc_pen = 0.0;
    // one float64 division per flagged neighbour instead of three (1 / (eng - sep) once per call, 1 / |r| once per neighbour):
    // <= 1 ulp from the quotients, far inside the reward's 1e-5 tolerance; the function was 15 % of this kernel's stall
    // samples in the airtaxi benchmark (profiles/r02_d_by_line_agent_cfg3.txt)
    const double inv_span = 1.0 / (eng - sep);
    for (int a = 0; a < N; ++a) {
        if (!((mask >> a) & 1u)) continue;
        const double2 pa = R.pos[a];
        const double rx = pa.x - x, ry = pa.y - y;
        const double dx = x - pa.x, dy = y - pa.y;
        const double rd = sqrt(dx * dx + dy * dy);
        const double closeness = 1.0 - clipd((rd - sep) * inv_span, 0.0, 1.0);
        // unit vector towards the other agent: (cos, sin)(atan2(ry, rx)) == (rx, ry) / |r| to ~1e-16 (reward tolerance
        // 1e-5); atan2(0, 0) = 0 for coincident agents. Three libm calls per flagged neighbour were 31 % of this kernel's
        // instructions in the airtaxi benchmark (profiles/r01_v7_*).
        const double inv_rd = 1.0 / rd;
        const double cdir = rd > 0.0 ? rx * inv_rd : 1.0, sdir = rd > 0.0 ? ry * inv_rd : 0.0;
        const double2 va = R.vel[(a < ai ? N : 0) + a];
        double change = cdir * (va.x - vpx) + sdir * (va.y - vpy);
        change = fabs(pymin(0.0, change));
        pc_pen += change * closeness;
    }
    return pc_pen;
}

// reward_hj_value (navigation_graph_safe.py:830-837, core.py:459-468)
template <int DYN, int N, int L, int O, bool F32>
__device__ __noinline__ double hj_value_reward(const GridDev* __restrict__ vg, const EmitRec<DYN, N, L, O>& R,
                                              const AgentScratch<DYN, N, L>& P, int ai, double x, double y, double sep, double cvalue_rew) {
    const GridDev& g = *vg;
    double r = 0.0;
    for (int a = 0; a < N; ++a) {
        if (a == ai) continue;
        const int adone = a < ai ? R.done[1][a] : R.done[0][a];
        if (adone) continue;
        // as2/as3 hold the pre-update states
        const double2 pa = R.pos[a];
        const double v = shift_value(pair_value_raw<DYN, F32>(g, x, y, P.as2[ai], P.as3[ai], pa.x, pa.y, P.as2[a], P.as3[a]), sep, g);
        const double cvp = fabs(pymin(v - 0.4, 0.0));
        r += cvalue_rew * cvp;
    }
    return r;
}

// ---------------------------------------------------------------------------------------------
// K_b: per-agent physics. A warp owns EPW <= 32 / N consecutive environments, N lanes each.
// ---------------------------------------------------------------------------------------------
// Episode summary of a resetting environment (graphworker, env_wrappers.py:861-874 + Scenario.info_callback's episode
// statistics): means over the env's N agents. Runs once per episode, so it lives OUT of the per-agent kernel's
// instruction stream (whole warp calls it; lanes of envs that do not reset take part in the shuffles only).
template <int N>
__device__ __noinline__ void episode_summary(const KParams& kp, int le, int env, bool write, int ep_len, double ep_travel_dist,
                                            int ep_done, int reached, int ep_conflict, int ep_multi, double ep_min_dist) {
    const lsm_config& c = kp.c;
    double s_len = 0, s_dist = 0, s_done = 0, s_reached = 0, s_conf = 0, s_min = 0, s_multi = 0, mn = INFINITY;
    const double len_i = ep_len == 0 ? 1.0 : (double)ep_len;
#pragma unroll 1
    for (int k = 0; k < N; ++k) {
        const int src = (le * N + k) & 31;
        s_len += (double)__shfl_sync(0xffffffffu, ep_len, src);
        s_dist += __shfl_sync(0xffffffffu, ep_travel_dist, src);
        s_done += (double)__shfl_sync(0xffffffffu, ep_done, src);
        s_reached += (double)__shfl_sync(0xffffffffu, reached, src);
        s_conf += __shfl_sync(0xffffffffu, (double)ep_conflict / len_i, src);
        s_multi += __shfl_sync(0xffffffffu, (double)ep_multi / len_i, src);
        const double md = __shfl_sync(0xffffffffu, ep_min_dist, src);
        s_min += md;
        if (md < mn) mn = md;
    }
    if (write) {
        double* out = kp.b.ep_info + (size_t)env * LSM_EP_COUNT;
        out[LSM_EP_TRAVEL_TIME_MEAN] = c.dt * (s_len / N);
        out[LSM_EP_TRAVEL_DISTANCE_MEAN] = s_dist / N;
        out[LSM_EP_DONE_PERCENTAGE] = s_done / N;
        out[LSM_EP_NUM_REACHED_GOAL_MEAN] = s_reached / N;
        out[LSM_EP_CONFLICT_PERCENTAGE] = s_conf / N;
        const double mm = s_min / N;
        out[LSM_EP_MIN_DISTANCE_MEAN] = isinf(mm) ? c.coordination_range : mm;
        out[LSM_EP_MIN_DISTANCE_MIN] = isinf(mn) ? c.coordination_range : mn;
        out[LSM_EP_MULTIPLE_ENGAGEMENT_PERCENTAGE] = s_multi / N;
    }
}

// F32 = LSM_FLAG_INTERP_FLOAT32: every grid lookup (filter gradient, airtaxi TTR term, in-kernel pair values, HJ_VALUE
// reward) in float32 arithmetic. A compile-time choice: this kernel is bound by instruction fetch, and unused flag code
// compiled into it costs time (DESIGN.md 3).
template <int DYN, int N, int L, int O, int BLOCK, int MINB, bool F32>
__global__ void __launch_bounds__(BLOCK, MINB) lsm_agent_kernel(const __grid_constant__ KParams kp) {
    using REC = EmitRec<DYN, N, L, O>;
    using SCR = AgentScratch<DYN, N, L>;
    constexpr int M = REC::M, E = REC::E;
    constexpr int G = N;                          // lanes per environment: 32 / N environments per warp, no padding lanes
    constexpr int Dobs = DYN == LSM_DYN_DOUBLE_INTEGRATOR ? 7 : 6;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const lsm_config& c = kp.c;
    const int lane = threadIdx.x & 31;
    const int warp_in_block = threadIdx.x >> 5;
    const int warps_per_block = blockDim.x >> 5;
    const int EPW = kp.EPW;                       // launch choice, 1 .. 32/G
    const int n = (int)kp.b.num_envs;
    const int le = lane / G;
    const int ai = lane - le * G;
    // this warp's records: EPW emit records (contiguous: dumped to global memory in one run), then EPW scratch blocks
    unsigned char* const wbase = smem_raw + (size_t)warp_in_block * EPW * (sizeof(REC) + sizeof(SCR));
    REC* const Rw = reinterpret_cast<REC*>(wbase);
    SCR* const Pw = reinterpret_cast<SCR*>(wbase + (size_t)EPW * sizeof(REC));
    const bool lane_has_env = le < EPW;
    REC& R = Rw[lane_has_env ? le : 0];
    SCR& P = Pw[lane_has_env ? le : 0];
    const unsigned group_mask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << ((le * G) & 31));
    const bool use_filter_arg = (c.flags & LSM_FLAG_USE_SAFETY_FILTER) != 0;
    const int ngroups = kp.ngroups;               // ceil(n / EPW), from the host
    const size_t fstride = (size_t)n * N;         // elements between two fields of the agent SoA
    pdl_launch_dependents();
    pdl_wait();
    tl_start(kp.timeline, TL_AGENT_START);

    for (int grp = kp.grp_begin + blockIdx.x * warps_per_block + warp_in_block; grp < ngroups; grp += gridDim.x * warps_per_block) {
        const int env0 = grp * EPW;
        const int env = env0 + le;
        bool env_on = lane_has_env && env < n;
        if (kp.mode == MODE_RESET && kp.env_mask != nullptr && env_on) env_on = kp.env_mask[env] != 0;
        const bool agent_on = env_on && ai < N;
        if (__ballot_sync(0xffffffffu, env_on) == 0u) continue;
        const int nenv = (n - env0) < EPW ? (n - env0) : EPW;   // envs of this group

        // ---------------- P0: load ----------------
        // everything this warp will touch later is requested now, so that the chain below pays ONE DRAM round trip
        if (agent_on) {
            const size_t a = (size_t)env * N + ai;
            if (kp.mode == MODE_STEP) {
                if (kp.action_idx != nullptr) prefetch_l2(kp.action_idx + a);
                else { prefetch_l2(kp.action_onehot + a * LSM_NUM_ACTIONS); prefetch_l2(kp.action_onehot + a * LSM_NUM_ACTIONS + LSM_NUM_ACTIONS - 1); }
                if (kp.pairval != nullptr) {
#pragma unroll
                    for (int k = 0; k < N * 8; k += 128) prefetch_l2(kp.pairval + a * N + k / 8);
                }
            }
            const double* afp = kp.b.agent_f64 + a;
            prefetch_l2(afp + LSM_AF_TIMES_REQ_A * fstride); prefetch_l2(afp + LSM_AF_TIMES_REQ_B * fstride);
            prefetch_l2(afp + LSM_AF_DISTS_GOAL_A * fstride); prefetch_l2(afp + LSM_AF_DISTS_GOAL_B * fstride);
            if (kp.mode == MODE_STEP) {   // read late (load_motion / load_bookkeeping)
                prefetch_l2(afp + LSM_AF_P_DIST * fstride); prefetch_l2(afp + LSM_AF_STATE_TIME * fstride);
                prefetch_l2(afp + LSM_AF_GOAL_MIN_TIME * fstride); prefetch_l2(afp + LSM_AF_DIST_LEFT * fstride);
                prefetch_l2(afp + LSM_AF_EP_TRAVEL_DIST * fstride); prefetch_l2(afp + LSM_AF_EP_MIN_DIST * fstride);
                const int* aipp = kp.b.agent_i32 + a;
                prefetch_l2(aipp + LSM_AI_NUM_COLLISIONS * fstride); prefetch_l2(aipp + LSM_AI_EP_TRAVEL_LEN * fstride);
                prefetch_l2(aipp + LSM_AI_EP_CONFLICT * fstride); prefetch_l2(aipp + LSM_AI_EP_MULTI * fstride);
                prefetch_l2(aipp + LSM_AI_EP_DONE * fstride);
            }
        }
        {
            const size_t lstride = (size_t)n * M;
            const double* src = kp.b.landmarks + (size_t)env0 * M;
            for (int idx = lane * 16; idx < nenv * M; idx += 32 * 16) {      // one request per 128-byte line and field
#pragma unroll
                for (int f = 0; f < LSM_LF_COUNT; ++f) {
                    prefetch_l2(src + f * lstride + idx);
                    prefetch_l2(src + f * lstride + (idx + 15 < nenv * M ? idx + 15 : nenv * M - 1));   // runs are not line aligned
                }
            }
        }
        double x = 0, y = 0, s2 = 0, s3 = 0, p_dist = 0, state_time = 0, min_rel = INFINITY, goal_min_time = INFINITY;
        double times_req = -1, dists_goal = -1, dist_left = -1, ep_travel_dist = 0, ep_min_dist = INFINITY, action_diff = 0;
        int reached = 0, done = 0, safety_filtered = 0, deconflict = -1, ncoll = 0;
        int ep_len = 0, ep_conflict = 0, ep_multi = 0, ep_done = 0;
        int nobst = 0;                            // world.num_obstacle_collisions (O > 0 only)
        int current_step = 0, reset_count = 0, parity = 0;
        double ratio = 0.0;
        double* const af = kp.b.agent_f64 + ((size_t)env * N + ai);
        int* const aip = kp.b.agent_i32 + ((size_t)env * N + ai);
        if (env_on) {
            current_step = kp.b.env_i32[(size_t)LSM_EI_CURRENT_STEP * n + env];
            reset_count = kp.b.env_i32[(size_t)LSM_EI_RESET_COUNT * n + env];
            parity = kp.b.env_i32[(size_t)LSM_EI_PARITY * n + env];
            ratio = kp.b.env_f64[(size_t)LSM_EF_CURRICULUM_RATIO * n + env];
        }
        if (agent_on) {
            x = af[LSM_AF_X * fstride]; y = af[LSM_AF_Y * fstride]; s2 = af[LSM_AF_S2 * fstride]; s3 = af[LSM_AF_S3 * fstride];
            reached = aip[LSM_AI_REACHED * fstride]; done = aip[LSM_AI_DONE * fstride];
            safety_filtered = aip[LSM_AI_SAFETY_FILTERED * fstride]; deconflict = aip[LSM_AI_DECONFLICT_IDX * fstride];
        }
        // Bookkeeping state is loaded where it is first needed (L2 hits after the prefetch above) instead of being
        // carried in registers through the filter / dynamics phase, whose register peak decides the occupancy.
#define LSM_LOAD_MOTION()  /* before the dynamics */ \
        if (agent_on) { p_dist = af[LSM_AF_P_DIST * fstride]; state_time = af[LSM_AF_STATE_TIME * fstride]; }
#define LSM_LOAD_BOOKKEEPING(STEP_MODE)  /* a step always overwrites min_rel / action_diff */ \
        if (agent_on) { \
            if (!(STEP_MODE)) { min_rel = af[LSM_AF_MIN_REL_DIST * fstride]; action_diff = af[LSM_AF_ACTION_DIFF * fstride]; } \
            goal_min_time = af[LSM_AF_GOAL_MIN_TIME * fstride]; \
            times_req = af[(parity ? LSM_AF_TIMES_REQ_B : LSM_AF_TIMES_REQ_A) * fstride]; \
            dists_goal = af[(parity ? LSM_AF_DISTS_GOAL_B : LSM_AF_DISTS_GOAL_A) * fstride]; \
            dist_left = af[LSM_AF_DIST_LEFT * fstride]; ep_travel_dist = af[LSM_AF_EP_TRAVEL_DIST * fstride]; \
            ep_min_dist = af[LSM_AF_EP_MIN_DIST * fstride]; \
            ncoll = aip[LSM_AI_NUM_COLLISIONS * fstride]; ep_len = aip[LSM_AI_EP_TRAVEL_LEN * fstride]; \
            ep_conflict = aip[LSM_AI_EP_CONFLICT * fstride]; ep_multi = aip[LSM_AI_EP_MULTI * fstride]; \
            ep_done = aip[LSM_AI_EP_DONE * fstride]; \
            if constexpr (O > 0) nobst = aip[LSM_AI_NUM_OBST_COLLISIONS * fstride]; \
        }
        if (kp.mode != MODE_STEP) { LSM_LOAD_MOTION() LSM_LOAD_BOOKKEEPING(false) }
        // landmark tables of the group's environments: contiguous runs per field
        {
            const int total = nenv * M;
            const size_t lstride = (size_t)n * M;
            const double* src = kp.b.landmarks + (size_t)env0 * M;
            for (int idx = lane; idx < total; idx += 32) {
                const int el = idx / M, m = idx - el * M;
                const double lxv = src[LSM_LF_X * lstride + idx], lyv = src[LSM_LF_Y * lstride + idx];
                const double lhv = src[LSM_LF_HEADING * lstride + idx], lsv = src[LSM_LF_SPEED * lstride + idx];
                const double sv = src[LSM_LF_SIN * lstride + idx], cv = src[LSM_LF_COS * lstride + idx];
                Rw[el].pos[N + m] = make_double2(lxv, lyv);
                SCR& T = Pw[el];
                T.lh[m] = lhv; T.lsp[m] = lsv; T.lsin[m] = sv; T.lcos[m] = cv;
                Rw[el].cst[m] = make_float4((float)sv, (float)cv, (float)lsv, 1.0f);   // landmark rows: type 1
            }
        }
        if constexpr (O > 0) {     // obstacle positions [2][n][O] of the group's environments; constant node columns
            for (int idx = lane; idx < nenv * O; idx += 32) {
                const int el = idx / O, k = idx - el * O;
                const double ox = kp.b.obstacles[((size_t)0 * n + (env0 + el)) * O + k], oy = kp.b.obstacles[((size_t)1 * n + (env0 + el)) * O + k];
                Rw[el].pos[N + M + k] = make_double2(ox, oy);
                Rw[el].cst[M + k] = make_float4(0.0f, 1.0f, 0.0f, 2.0f);
            }
        }
        Curriculum q = curriculum(kp, ratio);
        const int lvl = (int)(q.stair * 4.0);     // curriculum stair level: index of the squared-threshold tables
        if (agent_on) {
            R.pos[ai] = make_double2(x, y); P.as2[ai] = s2; P.as3[ai] = s3;
            R.done[0][ai] = done; R.reached[0][ai] = reached;
            if (ai == 0) { P.cur_sep = q.sep; P.cur_filter = q.world_filter ? 1 : 0; R.vel[2 * N] = make_double2(0.0, 0.0); }
        }
        __syncwarp();

        bool all_done_env = false;
        const unsigned any_filter = __ballot_sync(0xffffffffu, env_on && q.world_filter);
        int goal_obs = 0;                         // landmark index of the goal the env-level observation uses

        if (kp.mode == MODE_STEP) {
            // ---------------- P1: action decode, safety filter, dynamics ----------------
            current_step += 1;
            double raw0 = 0.0, raw1 = 0.0;
            if (agent_on) {
                int idx;
                if (kp.action_idx != nullptr) idx = kp.action_idx[(size_t)env * N + ai];
                else {   // np.argmax over the one-hot row: first maximum
                    const float* row = kp.action_onehot + ((size_t)env * N + ai) * LSM_NUM_ACTIONS;
                    idx = 0; float best = row[0];
                    for (int k = 1; k < LSM_NUM_ACTIONS; ++k) { const float v = row[k]; if (v > best) { best = v; idx = k; } }
                }
                const int i0 = idx / 5, i1 = idx - i0 * 5;
                raw0 = c.act_tab0[i0]; raw1 = c.act_tab1[i1];
                P.rawx[ai] = raw0; P.rawy[ai] = raw1;
            }
            __syncwarp();
            double safe0 = raw0, safe1 = raw1;
            LSM_LOAD_MOTION()
            // airtaxi: sin / cos of the own heading, evaluated once per internal step and shared by the filter's relative
            // frame (before the dynamics), the integration and the velocity / observation frame (after it)
            double hsc[2] = { 0.0, 1.0 };
            if constexpr (DYN != LSM_DYN_DOUBLE_INTEGRATOR) { if (agent_on) lsm_sincos_inl(s2, &hsc[0], &hsc[1]); }
            for (int it = 0; it < c.num_internal_step; ++it) {
                // HJ values of (ego, other): from lsm_pair_kernel for the states this launch started with, in-kernel
                // for later internal steps
                const bool precomputed = it == 0 && kp.pairval != nullptr;
                if (any_filter != 0u && !precomputed) {
                    pair_phase<DYN, N, L, O, F32>(&kp.vg, Rw, Pw, nenv, lane);
                    __syncwarp();
                }
                if (agent_on && q.world_filter) {
                    // np.argmin over the others (first minimum, ascending agent index), then resolve
                    int filt = 0, dec = -1;
                    safe0 = raw0; safe1 = raw1;
                    if (!done) {
                        double best_d2 = 0.0, best_v = 0.0; int kd = -1, kv = -1;
                        const double* pv = kp.pairval + ((size_t)env * N + ai) * N;
                        double vj[N];
#pragma unroll
                        for (int j = 0; j < N; ++j) {
                            vj[j] = INFINITY;
                            if (j == ai || R.done[0][j]) continue;
                            vj[j] = precomputed ? pv[j] : P.fval[ai * N + j];
                        }
#pragma unroll
                        for (int j = 0; j < N; ++j) {
                            if (j == ai || R.done[0][j]) continue;
                            const double2 pj = R.pos[j];
                            const double ddx = pj.x - x, ddy = pj.y - y;
                            const double d2 = ddx * ddx + ddy * ddy;
                            const double v = precomputed ? shift_value(vj[j], q.sep, kp.vg) : vj[j];
                            if (kd < 0 || d2 < best_d2) { kd = j; best_d2 = d2; }
                            if (kv < 0 || v < best_v) { kv = j; best_v = v; }
                        }
                        if (kv >= 0) {
                            dec = kv;
                            // `min distance > coordination_range` as an exact test on the squared distance
                            const double best_d = (best_d2 >= kp.r2_gt) ? INFINITY : 0.0;
                            const double2 po = R.pos[kv];
                            filter_resolve<DYN, true, F32>(kp, best_d, best_v, !isinf(best_v), x, y, s2, s3, po.x, po.y, P.as2[kv], P.as3[kv],
                                                           raw0, raw1, P.rawx[kv], P.rawy[kv], safe0, safe1, filt, hsc[0], hsc[1]);
                        }
                    }
                    deconflict = dec; safety_filtered = filt;
                }
                __syncwarp();   // everyone has read the pre-integration states
                if (agent_on) {
                    const double d0 = raw0 - safe0, d1 = raw1 - safe1;
                    action_diff = sqrt(d0 * d0 + d1 * d1);
                    if (!done) integrate<DYN>(x, y, s2, s3, safe0, safe1, c.dt, p_dist, state_time,
                                              DYN != LSM_DYN_DOUBLE_INTEGRATOR ? hsc : nullptr);
                    R.pos[ai] = make_double2(x, y); P.as2[ai] = s2; P.as3[ai] = s3;
                }
                __syncwarp();
            }
            // ---------------- P2: goal / reward / done ----------------
            int goal_pre = 0, goal_post = 0, reached_post = reached, done_post = done;
            double rew = 0.0;
            double vpx = 0, vpy = 0, vqx = 0, vqy = 0;
            double theta = 0, speed = 0;
            double cth = 1.0, sth = 0.0;
            bool reached_now = false;
            bool frozen = false;                  // reached its last goal this step: velocity / speed zeroed
            if (agent_on) {
                // the two / three trigonometric evaluations on this kernel's critical path are the force-inlined flavours
                // of the shared implementation (same arithmetic as lsm_atan2 / lsm_cos / lsm_sincos, include/lsm_math.h)
                speed = speed_of<DYN>(s2, s3);
                if constexpr (DYN == LSM_DYN_DOUBLE_INTEGRATOR) { theta = lsm_atan2_inl(s3, s2); vpx = s2; vpy = s3; }
                else { theta = s2; sth = hsc[0]; cth = hsc[1]; vpx = s3 * cth; vpy = s3 * sth; R.air.cth[ai] = cth; R.air.sth[ai] = sth; }   // hsc = lsm_sincos(s2)
                goal_pre = goal_index(reached, ai, N, M);
                const double2 gp = R.pos[N + goal_pre];
                const double gx = gp.x, gy = gp.y, gh = P.lh[goal_pre], gs = P.lsp[goal_pre];
                emit_obs_row<DYN, N, L, O>(R, P, ai, goal_pre, x, y, s2, s3, kp.b.obs + ((size_t)env * N + ai) * Dobs);
                // reward_reach_goal: navigation_graph_safe.py:691-791
                const double he = 0.5 - 0.5 * lsm_cos_inl(theta - gh);     // direction_alignment_error, utils.py:79-81
                const double hpr = 1.0 - clipd(he / q.heading_thresh, 0.0, 1.0);
                const double se = fabs(speed - gs);
                const double sen = clipd(se / q.speed_thresh, 0.0, 1.0);
                double cra = ratio_sloped(ratio, 0.25, 0.75);
                if (use_filter_arg) cra = 1.0;
                reached_now = goal_reached_he<DYN>(x, y, he, speed, gx, gy, gs, q);
                // The goal branches below run in a few warps of every step, and the kernel ends with its slowest warp.
                // Their trigonometry is inlined so that those warps do not wait on the fetch of cold out-of-line code.
                if (reached_now) {
                    double st = sth, ct = cth;          // airtaxi: lsm_sincos(theta) already
                    if constexpr (DYN == LSM_DYN_DOUBLE_INTEGRATOR) lsm_sincos_inl(theta, &st, &ct);
                    const double pr = goal_reward_factor(st, ct, gx - x, gy - y, hpr, sen);
                    double goal_rew;
                    if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) goal_rew = c.goal_rew * pr;
                    else goal_rew = c.goal_rew * (pr * cra + (1.0 - cra));
                    if (!done) rew += goal_rew;
                }
                if (!done) {
                    if constexpr (DYN == LSM_DYN_DOUBLE_INTEGRATOR) {
                        if (!use_filter_arg) rew -= magnetic_penalty(x, y, s2, s3, gx, gy, gh, gs, q.dist_thresh, q.sloped);
                        if (use_filter_arg) rew -= 1.0; else rew -= 1.0 * q.sloped;
                    } else {
                        double rpx, rpy;
                        rotate_into(x - gx, y - gy, P.lcos[goal_pre], P.lsin[goal_pre], rpx, rpy);   // tabulated cos / sin(gh)
                        const double rs[4] = { rpx, rpy, theta - gh, speed };
                        double ttr = grid_value<4, F32>(kp.tg, rs);
                        if (isnan(ttr)) ttr = kp.tg.ttr_max;
                        rew -= 0.04 * ttr;
                        rew -= sen * cra;
                    }
                }
                // update_reached_goal_and_done (+ freeze_agent): navigation_graph_safe.py:658-675, 1091-1099
                if (reached_now && !done) reached_post = reached + 1;
                done_post = done;
                vqx = vpx; vqy = vpy;
                double s2q = s2, s3q = s3;
                if (reached_post >= L) {
                    done_post = 1; frozen = true;
                    if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) { s2q = 0.0; s3q = 0.0; vqx = 0.0; vqy = 0.0; }
                    else { s3q = 0.0; vqx = s3q * cth; vqy = s3q * sth; }
                }
                goal_post = goal_index(reached_post, ai, N, M);
                R.vel[ai] = make_double2(vpx, vpy); R.vel[N + ai] = make_double2(vqx, vqy);
                R.pos[E + ai] = gp; R.pos[E + N + ai] = R.pos[N + goal_post];
                { float4 t = R.cst[goal_pre]; t.w = 0.0f; R.cst[REC::CA + ai] = t; }
                { float4 t = R.cst[goal_post]; t.w = 0.0f; R.cst[REC::CA + N + ai] = t; }
                if constexpr (DYN != LSM_DYN_DOUBLE_INTEGRATOR) {
                    R.air.spd_post[ai] = s3q; R.air.goal[0][ai] = goal_pre; R.air.goal[1][ai] = goal_post;
                }
                R.reached[1][ai] = reached_post; R.done[1][ai] = done_post;
                // as2/as3 keep the PRE-update state (the HJ_VALUE term of later agents only reads agents that are
                // not done, whose pre and post states coincide); the lane's registers take the post state
                s2 = s2q; s3 = s3q;
            }
            __syncwarp();
            LSM_LOAD_BOOKKEEPING(true)
            if (agent_on) {
                // one pass over the other agents: min distance, collisions, episode statistics, proximity rewards.
                // Agent a is seen after its own update if a < i (rewards) / a <= i (statistics), else before.
                double mind2 = INFINITY;                       // core.py:696-709
                double stat_mind2 = INFINITY; int cnt = 0;      // environment.py:1004-1022
                double r_sv = 0.0;                              // navigation_graph_safe.py:793-798
                int pc_count = 0;                               // navigation_graph_safe.py:800-823
                const bool want_sv = (c.flags & LSM_FLAG_SAFETY_VIOLATION) != 0;
                const bool want_pc = (c.flags & LSM_FLAG_POTENTIAL_CONFLICT) != 0;
                unsigned pc_mask = 0u;
                // airtaxi: the loop stays rolled (-5 % code in a kernel bound by instruction fetch: cfg3 0.3385 -> 0.3348 ms, same-box
                // A/B); the double-integrator kernels measure the same either way and keep the unrolled loop
                constexpr int kOthersUnroll = DYN == LSM_DYN_DOUBLE_INTEGRATOR ? N : 1;
#pragma unroll kOthersUnroll
                for (int a = 0; a < N; ++a) {
                    if (a == ai) continue;
                    // squared distance after the dynamics; (p_i - p_a)^2 == (p_a - p_i)^2 exactly, so both lanes of a
                    // pair see the same value (core.py:514-543)
                    const double2 pa = R.pos[a];
                    const double dx = x - pa.x, dy = y - pa.y;
                    const double d2 = dx * dx + dy * dy;
                    const int apre = R.done[0][a], apost = R.done[1][a];
                    if (!done && !apre && d2 < mind2) mind2 = d2;
                    if (d2 < kp.col2_lt) ncoll += 1;           // navigation_graph_safe.py:405-413, 497-501
                    const int adone_r = a < ai ? apost : apre;
                    if (want_sv && d2 < kp.sep2_lt[lvl] && !adone_r) r_sv += q.conflict_rew;
                    if (want_pc && d2 < kp.eng2_lt[lvl] && !adone_r) { pc_mask |= 1u << a; pc_count += 1; }
                    const int adone_s = a <= ai ? apost : apre;
                    if (!adone_s && d2 < kp.r2_lt && d2 > 0.0) {
                        if (d2 < kp.engref2_lt) cnt++;
                        if (d2 < stat_mind2) stat_mind2 = d2;
                    }
                }
                if constexpr (O > 0) {      // info_callback, navigation_graph_safe.py:402-404, 452-465: any obstacle within 1.05 * (size + size)
                    bool hit = false;
                    for (int k = 0; k < O; ++k) {
                        const double2 po = R.pos[N + M + k];
                        const double dx = po.x - x, dy = po.y - y;
                        hit = hit || (dx * dx + dy * dy < kp.col2_lt);
                    }
                    if (hit) nobst += 1;
                }
                min_rel = sqrt(mind2);
                if (want_sv) rew += r_sv;
                if (pc_count > 1)
                    rew += q.multi_rew * potential_conflict_penalty<DYN, N, L, O>(R, pc_mask, ai, x, y, vpx, vpy, q.sep, q.eng);
                if ((c.flags & LSM_FLAG_DIFF_FROM_FILTERED_ACTION) && use_filter_arg) {   // :825-828
                    if (!done) rew += q.diff_rew * action_diff;
                }
                if (c.flags & LSM_FLAG_HJ_VALUE)
                    rew += hj_value_reward<DYN, N, L, O, F32>(&kp.vg, R, P, ai, x, y, q.sep, q.cvalue_rew);
                rew = clipd(rew, c.min_reward, c.max_reward);
                if (!done_post) {
                    ep_len += 1;
                    ep_travel_dist += norm2(vqx, vqy) * c.dt;
                    if (stat_mind2 < INFINITY) {
                        if (cnt > 1) ep_multi += 1;
                        if (stat_mind2 < kp.septgt2_lt) ep_conflict += 1;
                        const double mn = sqrt(stat_mind2);
                        if (mn < ep_min_dist) ep_min_dist = mn;
                    }
                }
                if (done_post) ep_done = 1;
                // info_callback state: navigation_graph_safe.py:386-413 (post-update goal and velocity)
                if (times_req == -1.0) {
                    // once times_required is set all three fields are frozen, so the goal test is only needed here
                    const double2 gq = R.pos[N + goal_post];
                    const double dx = x - gq.x, dy = y - gq.y;
                    // same goal and same (unfrozen) state as before the update -> same answer as `reached_now`
                    bool r2 = reached_now;
                    if (goal_post != goal_pre || done_post != done) {
                        // theta_of / speed_of of the post-update state: unchanged unless the double integrator was frozen
                        // to zero velocity (lsm_atan2(+0, +0) = +0, sqrt(0) = 0); the airtaxi keeps its heading
                        const bool zero = DYN == LSM_DYN_DOUBLE_INTEGRATOR && frozen;
                        const double th2 = zero ? 0.0 : theta;
                        const double sp2 = DYN == LSM_DYN_DOUBLE_INTEGRATOR ? (zero ? 0.0 : speed) : s3;
                        const double he2 = 0.5 - 0.5 * lsm_cos_inl(th2 - P.lh[goal_post]);   // direction_alignment_error
                        r2 = goal_reached_he<DYN>(x, y, he2, sp2, gq.x, gq.y, P.lsp[goal_post], q);
                    }
                    if (r2) times_req = (double)current_step * c.dt;
                    dists_goal = p_dist; dist_left = sqrt(dx * dx + dy * dy);
                }
            }
            if (agent_on && kp.b.reward_individual != nullptr) kp.b.reward_individual[(size_t)env * N + ai] = (float)rew;
            if (c.flags & LSM_FLAG_SHARED_REWARD) {     // environment.py:1032-1037, sequential sum in agent order
                double s = 0.0;
#pragma unroll
                for (int k = 0; k < N; ++k) s += __shfl_sync(0xffffffffu, rew, (le * G + k) & 31);
                rew = s;
            }
            const bool done_out = done_post || (current_step >= c.episode_length);   // environment.py:260-268
            const unsigned not_done = __ballot_sync(0xffffffffu, agent_on && !done_out);
            all_done_env = env_on && ((not_done & group_mask) == 0u);
            if (agent_on) {
                kp.b.reward[(size_t)env * N + ai] = (float)rew;
                kp.b.done[(size_t)env * N + ai] = (uint8_t)done_out;
                reinterpret_cast<double2*>(kp.b.safe_action)[(size_t)env * N + ai] = make_double2(safe0, safe1);
            }
            reached = reached_post; done = done_post;
            parity ^= 1;
        } else {
            if (agent_on) {
                double vx, vy;
                if constexpr (DYN == LSM_DYN_DOUBLE_INTEGRATOR) { vx = s2; vy = s3; }
                else { double ct, st; lsm_sincos(s2, &st, &ct); vx = s3 * ct; vy = s3 * st; R.air.cth[ai] = ct; R.air.sth[ai] = st; }
                const int g = goal_index(reached, ai, N, M);
                goal_obs = g;
                R.vel[ai] = make_double2(vx, vy); R.vel[N + ai] = make_double2(vx, vy);
                const double2 gp = R.pos[N + g];
                R.pos[E + ai] = gp; R.pos[E + N + ai] = gp;
                float4 cc = R.cst[g]; cc.w = 0.0f;
                R.cst[REC::CA + ai] = cc; R.cst[REC::CA + N + ai] = cc;
                if constexpr (DYN != LSM_DYN_DOUBLE_INTEGRATOR) {
                    R.air.spd_post[ai] = s3; R.air.goal[0][ai] = g; R.air.goal[1][ai] = g;
                }
                R.reached[1][ai] = reached; R.done[1][ai] = done;
            }
            __syncwarp();
        }

        // ---------------- P3: reset (graphworker auto-reset or explicit) ----------------
        const bool do_reset = (kp.mode == MODE_STEP && kp.flag && all_done_env) || (kp.mode == MODE_RESET && env_on);
        const bool sample = (kp.mode == MODE_STEP) ? true : (kp.flag != 0);
        const unsigned reset_lanes = __ballot_sync(0xffffffffu, do_reset);
        if (reset_lanes != 0u) {
            episode_summary<N>(kp, le, env, do_reset && ai == 0, ep_len, ep_travel_dist, ep_done, reached, ep_conflict, ep_multi,
                               ep_min_dist);
            if (do_reset && kp.mode == MODE_STEP && kp.b.term_f64 != nullptr) {
                // `parity` already names the slot this step's values go to; last step's are still in the other one
                if (agent_on)
                    term_snapshot(kp.b, (size_t)env * N + ai, fstride, x, y, min_rel, dist_left, times_req,
                                  af[(parity ? LSM_AF_TIMES_REQ_A : LSM_AF_TIMES_REQ_B) * fstride], dists_goal,
                                  af[(parity ? LSM_AF_DISTS_GOAL_A : LSM_AF_DISTS_GOAL_B) * fstride], goal_min_time, ncoll,
                                  safety_filtered);
                if constexpr (O > 0) { if (agent_on) kp.b.term_i32[(size_t)LSM_TI_NUM_OBST_COLLISIONS * fstride + (size_t)env * N + ai] = nobst; }
                if (ai == 0) kp.b.term_env_f64[env] = ratio;
            }
            if (do_reset) {
                current_step = 0;
                ratio = clipd((double)kp.episode / (double)c.num_total_episode, 0.0, 1.0);
                q = curriculum(kp, ratio);
            }
            if (do_reset && sample && ai == 0) sample_scenario<DYN, N, L, O>(kp, R, P, env, reset_count, ratio);
            __syncwarp();
            if (do_reset && agent_on) {
                if (sample) { const double2 p = R.pos[ai]; x = p.x; y = p.y; s2 = P.as2[ai]; s3 = P.as3[ai]; }
                done = 0; reached = 0;
                p_dist = 0.0; state_time = 0.0;
                const double2 g0 = R.pos[N + ai];
                goal_min_time = norm2(x - g0.x, y - g0.y) / c.agent_max_speed;   // navigation_graph_safe.py:525-535
                times_req = -1.0; dists_goal = -1.0; dist_left = -1.0; ncoll = 0; nobst = 0;
                ep_len = 0; ep_travel_dist = 0.0; ep_done = 0; ep_conflict = 0; ep_multi = 0; ep_min_dist = INFINITY;
                double vx, vy;
                if constexpr (DYN == LSM_DYN_DOUBLE_INTEGRATOR) { vx = s2; vy = s3; }
                else { double ct, st; lsm_sincos(s2, &st, &ct); vx = s3 * ct; vy = s3 * st; R.air.cth[ai] = ct; R.air.sth[ai] = st; }
                R.pos[ai] = make_double2(x, y); P.as2[ai] = s2; P.as3[ai] = s3;
                R.vel[ai] = make_double2(vx, vy); R.vel[N + ai] = make_double2(vx, vy);
                R.pos[E + ai] = g0; R.pos[E + N + ai] = g0;
                float4 cc = R.cst[ai]; cc.w = 0.0f;
                R.cst[REC::CA + ai] = cc; R.cst[REC::CA + N + ai] = cc;
                if constexpr (DYN != LSM_DYN_DOUBLE_INTEGRATOR) {
                    R.air.spd_post[ai] = s3; R.air.goal[0][ai] = ai; R.air.goal[1][ai] = ai;
                }
                R.reached[0][ai] = 0; R.reached[1][ai] = 0; R.done[0][ai] = 0; R.done[1][ai] = 0;
                emit_obs_row<DYN, N, L, O>(R, P, ai, ai, x, y, s2, s3, kp.b.obs + ((size_t)env * N + ai) * Dobs);
            }
            if (do_reset && sample) reset_count += 1;
            __syncwarp();
            if (sample) {
                const size_t lstride = (size_t)n * M;
                for (int el = 0; el < nenv; ++el) {
                    if (!((reset_lanes >> ((el * G) & 31)) & 1u)) continue;
                    const REC& T = Rw[el];
                    const SCR& U = Pw[el];
                    double* dst = kp.b.landmarks + (size_t)(env0 + el) * M;
                    for (int m = lane; m < M; m += 32) {
                        const double2 p = T.pos[N + m];
                        dst[LSM_LF_X * lstride + m] = p.x; dst[LSM_LF_Y * lstride + m] = p.y;
                        dst[LSM_LF_HEADING * lstride + m] = U.lh[m]; dst[LSM_LF_SPEED * lstride + m] = U.lsp[m];
                        dst[LSM_LF_SIN * lstride + m] = U.lsin[m]; dst[LSM_LF_COS * lstride + m] = U.lcos[m];
                    }
                    if constexpr (O > 0) {
                        for (int k = lane; k < O; k += 32) {
                            const double2 p = T.pos[N + M + k];
                            kp.b.obstacles[((size_t)0 * n + (env0 + el)) * O + k] = p.x;
                            kp.b.obstacles[((size_t)1 * n + (env0 + el)) * O + k] = p.y;
                        }
                    }
                }
            }
        } else if (kp.mode == MODE_OBSERVE && agent_on) {
            emit_obs_row<DYN, N, L, O>(R, P, ai, goal_obs, x, y, s2, s3, kp.b.obs + ((size_t)env * N + ai) * Dobs);
        }

        // ---------------- state write-back ----------------
        if (kp.mode != MODE_OBSERVE) {
            if (env_on && ai == 0) {
                kp.b.env_i32[(size_t)LSM_EI_CURRENT_STEP * n + env] = current_step;
                kp.b.env_i32[(size_t)LSM_EI_RESET_COUNT * n + env] = reset_count;
                kp.b.env_i32[(size_t)LSM_EI_PARITY * n + env] = parity;
                kp.b.env_i32[(size_t)LSM_EI_JUST_RESET * n + env] = do_reset ? 1 : 0;
                kp.b.env_f64[(size_t)LSM_EF_CURRICULUM_RATIO * n + env] = ratio;
            }
            if (agent_on) {
                af[LSM_AF_X * fstride] = x; af[LSM_AF_Y * fstride] = y; af[LSM_AF_S2 * fstride] = s2; af[LSM_AF_S3 * fstride] = s3;
                af[LSM_AF_P_DIST * fstride] = p_dist; af[LSM_AF_STATE_TIME * fstride] = state_time;
                af[LSM_AF_MIN_REL_DIST * fstride] = min_rel; af[LSM_AF_GOAL_MIN_TIME * fstride] = goal_min_time;
                af[(parity ? LSM_AF_TIMES_REQ_B : LSM_AF_TIMES_REQ_A) * fstride] = times_req;
                af[(parity ? LSM_AF_DISTS_GOAL_B : LSM_AF_DISTS_GOAL_A) * fstride] = dists_goal;
                if (do_reset) {
                    af[(parity ? LSM_AF_TIMES_REQ_A : LSM_AF_TIMES_REQ_B) * fstride] = times_req;
                    af[(parity ? LSM_AF_DISTS_GOAL_A : LSM_AF_DISTS_GOAL_B) * fstride] = dists_goal;
                }
                af[LSM_AF_DIST_LEFT * fstride] = dist_left; af[LSM_AF_EP_TRAVEL_DIST * fstride] = ep_travel_dist;
                af[LSM_AF_EP_MIN_DIST * fstride] = ep_min_dist; af[LSM_AF_ACTION_DIFF * fstride] = action_diff;
                aip[LSM_AI_REACHED * fstride] = reached; aip[LSM_AI_DONE * fstride] = done;
                aip[LSM_AI_SAFETY_FILTERED * fstride] = safety_filtered; aip[LSM_AI_DECONFLICT_IDX * fstride] = deconflict;
                aip[LSM_AI_NUM_COLLISIONS * fstride] = ncoll; aip[LSM_AI_EP_TRAVEL_LEN * fstride] = ep_len;
                aip[LSM_AI_EP_CONFLICT * fstride] = ep_conflict; aip[LSM_AI_EP_MULTI * fstride] = ep_multi;
                aip[LSM_AI_EP_DONE * fstride] = ep_done;
                if constexpr (O > 0) aip[LSM_AI_NUM_OBST_COLLISIONS * fstride] = nobst;
            }
        }
        // ---------------- emit records -> global memory (consumed by lsm_emit_kernel; L2 resident) ----------------
        if (env_on && ai == 0) R.next_filter = q.world_filter ? 1 : 0;     // q follows a reset's new curriculum ratio
        if constexpr (DYN != LSM_DYN_DOUBLE_INTEGRATOR) {
            if (agent_on) R.air.theta[ai] = s2;
            for (int idx = lane; idx < nenv * M; idx += 32) {
                const int el = idx / M, m = idx - el * M;
                Rw[el].air.lsin[m] = Pw[el].lsin[m]; Rw[el].air.lcos[m] = Pw[el].lcos[m]; Rw[el].air.lsp[m] = Pw[el].lsp[m];
            }
            if constexpr (O > 0) {     // obstacles: heading 0, speed 0
                for (int idx = lane; idx < nenv * O; idx += 32) {
                    const int el = idx / O, k = idx - el * O;
                    Rw[el].air.lsin[M + k] = 0.0; Rw[el].air.lcos[M + k] = 1.0; Rw[el].air.lsp[M + k] = 0.0;
                }
            }
        }
        __syncwarp();
        {
            constexpr int Q = (int)(sizeof(REC) / 16);
            const unsigned on_mask = __ballot_sync(0xffffffffu, env_on && ai == 0);
            for (int el = 0; el < nenv; ++el) {
                if (!((on_mask >> ((el * G) & 31)) & 1u)) continue;
                const int4* src = reinterpret_cast<const int4*>(&Rw[el]);
                int4* dst = reinterpret_cast<int4*>(kp.emit_rec + (size_t)(env0 + el) * sizeof(REC));
                for (int k = lane; k < Q; k += 32) dst[k] = src[k];
            }
            // placement 4: next step's HJ pair values from the records still in shared memory
            if (kp.pair_tail) pair_tail_phase<DYN, N, L, O, F32>(&kp.vg, Rw, kp.pairval, env0, nenv, on_mask, lane);
        }
        __syncwarp();
    }
    tl_end(kp.timeline, TL_AGENT_END);
}

// ---------------------------------------------------------------------------------------------
// K_c: graph observation (navigation_graph_safe.py:932-994 + utils.py:139-255). Persistent blocks of WPE warps
// loop over environments; the outputs of one environment (N adjacency matrices + N*E node rows, >= 96 % of the
// step's bytes) are assembled in shared memory and leave through TMA bulk copies, so the stores of environment k
// drain to HBM while environment k+1 is being computed. The next record is prefetched with cp.async.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(void* sdst, const void* gsrc) {
    const unsigned saddr = (unsigned)__cvta_generic_to_shared(sdst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(saddr), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

template <int DYN, int N, int L, int O>
struct EmitGeom {
    using REC = EmitRec<DYN, N, L, O>;
    static constexpr int E = REC::E, W = REC::W, EE = E * E;
    static constexpr int F = DYN == LSM_DYN_DOUBLE_INTEGRATOR ? 10 : 11;
    static constexpr int ROWS = N * E;
    // node rows leave in chunks of CR rows (<= 16 KB, CR % 4 == 0 so that the byte count is a multiple of 16)
    static constexpr int CR_MAX = (16384 / (F * 4)) / 4 * 4;
    static constexpr bool NODE_BULK = (ROWS % 4 == 0);
    static constexpr int CR = NODE_BULK ? (ROWS < CR_MAX ? ROWS : CR_MAX) : 32;
    static constexpr int NCHUNK = (ROWS + CR - 1) / CR;
    static constexpr bool ADJ_BULK = (EE % 4 == 0);             // 16-byte multiple per observer matrix
    // double-buffer the per-env tiles when they are small; one buffer (wait for the drain) when a tile is tens of KB
    // (airtaxi: 12 KB - measured at 10 agents, where one 17 KB tile and twice the resident blocks beat two tiles by 1-2 % of
    // the step, profiles/experiments/r02_emit_ablation_cfg3.txt; the 8-agent double integrator's 10 KB tile stays double-buffered)
    static constexpr int NBUF = (EE * 4 + CR * F * 4) <= (DYN == LSM_DYN_DOUBLE_INTEGRATOR ? 24 * 1024 : 12 * 1024) ? 2 : 1;
};

template <int DYN, int N, int L, int O, int WPE>
struct __align__(16) EmitShared {
    using GEO = EmitGeom<DYN, N, L, O>;
    using REC = EmitRec<DYN, N, L, O>;
    REC rec[2];                                              // current / prefetched record
    alignas(16) float dthr[GEO::NBUF][GEO::EE];              // radius-thresholded distance matrix (float32, what adj stores)
    alignas(16) float nodes[GEO::NBUF][GEO::CR * GEO::F];    // node-row chunk
    unsigned disc[2][GEO::W], keepm[N * GEO::W];
    unsigned sel[N * GEO::W];                                // KParams::sel_tab, read once per block (not once per environment)
    // fused COO edge output: non-zero bit mask of every row of the thresholded matrix, exclusive row offsets per observer
    unsigned rowmask[GEO::E * GEO::W];
    unsigned short rowoff[N * GEO::E];      // <= E * (E - 1): 36 672 at the largest shape lsm_create accepts (E = 192)
    static_assert(GEO::E * (GEO::E - 1) <= 65535, "rowoff holds an observer's edge count in 16 bits");
    long long gbase[N];
    long long range_base;
};

// Fused COO edge output of one environment (SURVEY 8f N2): kept OUT OF LINE so that its registers do not count against
// the occupancy of the dense path (69 -> 91 registers per thread when inlined, one resident block per SM fewer).
template <int DYN, int N, int L, int O, int WPE>
__device__ __noinline__ void emit_edges(EmitShared<DYN, N, L, O, WPE>& S, const KParams& kp, int ee, const float* dthr, bool uniform) {
    using GEO = EmitGeom<DYN, N, L, O>;
    constexpr int E = GEO::E, W = GEO::W;
    constexpr int T = 32 * WPE;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // `uniform`: no connectivity flag changed in this step, so every observer sees the SAME graph (the keep masks of all
    // observers are equal): row counts and row offsets are computed once (for observer 0) and shared.
    // (e0) where this environment's N graphs start in the global list: independent loads, one thread per observer, issued
    //      before anything else (lsm_edge_count_kernel left: prefix inside its block's env run + base of that block)
    for (int i = tid; i < N; i += T) {
        const long long gb = S.range_base + kp.edge_block_base[kp.edge_block_ofs + (ee - kp.env_begin) / kp.edge_envs_per_block] +
                             kp.edge_local[(size_t)ee * N + i];
        S.gbase[i] = gb;
        kp.edge_offsets[(size_t)ee * N + i] = gb;
    }
    // (e1) non-zero bit mask of every row (one ballot per 32 columns)
    for (int a = warp; a < E; a += WPE) {
#pragma unroll
        for (int w = 0; w < W; ++w) {
            const int b2 = w * 32 + lane;
            const unsigned m = __ballot_sync(0xffffffffu, b2 < E && dthr[a * E + b2] != 0.0f);
            if (lane == 0) S.rowmask[a * W + w] = m;
        }
    }
    __syncthreads();
    // (e2) edges of row a as observer i sees it, then the exclusive prefix over the rows of each observer
    const int NO = uniform ? 1 : N;
    for (int k = tid; k < NO * E; k += T) {
        const int i = k / E, a = k - i * E;
        int cnt = 0;
        if ((S.keepm[i * W + (a >> 5)] >> (a & 31)) & 1u) {
#pragma unroll
            for (int w = 0; w < W; ++w) cnt += __popc(S.rowmask[a * W + w] & S.keepm[i * W + w]);
        }
        S.rowoff[k] = (unsigned short)cnt;
    }
    __syncthreads();
    for (int i = warp; i < NO; i += WPE) {
        int running = 0;
        for (int c0 = 0; c0 < E; c0 += 32) {
            const int a = c0 + lane;
            const int v = a < E ? S.rowoff[i * E + a] : 0;
            int incl = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int t2 = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t2; }
            if (a < E) S.rowoff[i * E + a] = (unsigned short)(running + incl - v);
            running += __shfl_sync(0xffffffffu, incl, 31);
        }
    }
    __syncthreads();
    // (e3) fill. Dense graphs (mean degree > 8): one warp per (observer, row), lane = column inside a 32-column word,
    //      rank by popcount - coalesced stores. Sparse graphs: one LANE per (observer, row) walking the few set bits
    //      of its row (a warp per row would spend ~40 instructions on a row that holds two edges). A lane per ROW with an
    //      inner loop over the observers of a shared graph was slower (cfg4 / world 40: 2.07 vs 1.5 ms per step).
    {
        long long* const src = kp.edge_index;
        long long* const dst = kp.edge_index + kp.edge_capacity;
        const long long cap = kp.edge_capacity;
        const unsigned lt = (1u << lane) - 1u;
        // total edges of the env = last observer's end; mean degree decides the strategy (block-uniform)
        int env_edges = 0;
        for (int i = 0; i < N; ++i) env_edges += S.rowoff[(uniform ? 0 : i) * E + E - 1];          // lower bound is enough for the choice
        if (env_edges > 8 * N * E) {
            for (int r = warp; r < N * E; r += WPE) {
                const int i = r / E, a = r - i * E;
                if (!((S.keepm[i * W + (a >> 5)] >> (a & 31)) & 1u)) continue;
                const long long node0 = ((long long)ee * N + i) * E;
                long long p0 = S.gbase[i] + S.rowoff[uniform ? a : r];
#pragma unroll
                for (int w = 0; w < W; ++w) {
                    const unsigned m = S.rowmask[a * W + w] & S.keepm[i * W + w];
                    if ((m >> lane) & 1u) {
                        const long long p = p0 + __popc(m & lt);
                        if (p < cap) {
                            const int b2 = w * 32 + lane;
                            src[p] = node0 + a; dst[p] = node0 + b2; kp.edge_attr[p] = dthr[a * E + b2];
                        }
                    }
                    p0 += __popc(m);
                }
            }
        } else {
            for (int r = tid; r < N * E; r += T) {
                const int i = r / E, a = r - i * E;
                if (!((S.keepm[i * W + (a >> 5)] >> (a & 31)) & 1u)) continue;
                const long long node0 = ((long long)ee * N + i) * E;
                long long p = S.gbase[i] + S.rowoff[uniform ? a : r];
#pragma unroll
                for (int w = 0; w < W; ++w) {
                    unsigned m = S.rowmask[a * W + w] & S.keepm[i * W + w];
                    while (m != 0u) {
                        const int bit = __ffs(m) - 1;
                        m &= m - 1u;
                        if (p < cap) {
                            const int b2 = w * 32 + bit;
                            src[p] = node0 + a; dst[p] = node0 + b2; kp.edge_attr[p] = dthr[a * E + b2];
                        }
                        ++p;
                    }
                }
            }
        }
    }
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------
// graph emission from one record: shared by lsm_emit_kernel (every observer of an env) and lsm_record_emit_kernel (one
// observer of one stored record), so that both write the same bytes
// ---------------------------------------------------------------------------------------------
// float32 adjacency entry of an entity pair at squared distance d2: non-zero strictly inside the radius and above r2_nz
// (the non-zero value is at least ~1e-15: d2f >= 1e-30, so "adj_value != 0" is exactly that float64 test)
__device__ __forceinline__ float adj_value(double d2, double r2_lt, double r2_nz) {
    const float d2f = fmaxf((float)d2, 1.0e-30f);
    float rs;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(rs) : "f"(d2f));
    return (d2 < r2_lt && d2 > r2_nz) ? d2f * rs : 0.0f;
}

// entities one mask word of an observer keeps: an entity whose owner is <= the observer (sel) is seen after this step's
// goal update (disconnected after), any other before it
__device__ __forceinline__ unsigned keep_word(unsigned disc_post, unsigned disc_pre, unsigned sel) {
    return ~((disc_post & sel) | (disc_pre & ~sel));
}

// node-feature row r = i * E + e (observer i, entity e) of the record: F floats, or 7 with graph_feat_type 'global'
template <int DYN, int N, int L, int O>
__device__ __forceinline__ void node_feature_row(const EmitRec<DYN, N, L, O>& R, int r, bool gfeat, float* o) {
    using REC = EmitRec<DYN, N, L, O>;
    constexpr int M = REC::M, E = REC::E;
    const int i = r / E, e = r - i * E;
    const double2 pi = R.pos[i], vi = R.vel[N + i];
    const bool is_agent = e < N;
    const int sel = (e <= i) ? N : 0;     // agents <= i are seen after their own update
    const int vidx = is_agent ? sel + e : 2 * N;
    const int gidx = is_agent ? E + sel + e : e;
    const int cidx = is_agent ? REC::CA + sel + e : e - N;
    if (gfeat) {
        // an agent's goal is its FIRST landmark (optimal_match_index = arange, navigation_graph_safe.py:179), a
        // landmark's goal is itself; velocities are world-frame (landmarks: zero)
        const double2 pe = R.pos[e], ve = R.vel[vidx], ge = is_agent ? R.pos[N + e] : pe;
        o[0] = (float)ve.x; o[1] = (float)ve.y; o[2] = (float)pe.x; o[3] = (float)pe.y;
        o[4] = (float)ge.x; o[5] = (float)ge.y; o[6] = is_agent ? 0.0f : ((O == 0 || e < N + M) ? 1.0f : 2.0f);
        (void)gidx; (void)cidx; (void)pi; (void)vi;
    } else if constexpr (DYN == LSM_DYN_DOUBLE_INTEGRATOR) {
        // utils.py:201-255: [p_e - p_i, v_e - v_i, goal_e - p_i, sin gh, cos gh, gspeed, type]
        const double2 pe = R.pos[e], ve = R.vel[vidx], ge = R.pos[gidx];
        const float4 cc = R.cst[cidx];
        float2* o2 = reinterpret_cast<float2*>(o);   // rows are 40 B: 8 B aligned
        o2[0] = make_float2((float)(pe.x - pi.x), (float)(pe.y - pi.y));
        o2[1] = make_float2((float)(ve.x - vi.x), (float)(ve.y - vi.y));
        o2[2] = make_float2((float)(ge.x - pi.x), (float)(ge.y - pi.y));
        o2[3] = make_float2(cc.x, cc.y);
        o2[4] = make_float2(cc.z, cc.w);
    } else {
        const double ci = R.air.cth[i], si = R.air.sth[i];
        if (e < N) {
            const int g = R.air.goal[sel ? 1 : 0][e];
            const double2 pe = R.pos[e], ve = R.vel[vidx], ge = R.pos[gidx];
            double rx, ry, gx, gy;
            rotate_into(pe.x - pi.x, pe.y - pi.y, ci, si, rx, ry);
            rotate_into(ge.x - pi.x, ge.y - pi.y, ci, si, gx, gy);
            const double ce = R.air.cth[e], se = R.air.sth[e];
            o[0] = (float)rx; o[1] = (float)ry; o[2] = (float)norm2(ve.x - vi.x, ve.y - vi.y);
            o[3] = (float)(se * ci - ce * si); o[4] = (float)(ce * ci + se * si);
            o[5] = (float)gx; o[6] = (float)gy;
            o[7] = (float)(R.air.lsin[g] * ci - R.air.lcos[g] * si); o[8] = (float)(R.air.lcos[g] * ci + R.air.lsin[g] * si);
            o[9] = (float)R.air.lsp[g]; o[10] = 0.0f;
        } else {
            const int m = e - N;
            const double2 pe = R.pos[e];
            double rx, ry;
            rotate_into(pe.x - pi.x, pe.y - pi.y, ci, si, rx, ry);
            const float sh = (float)(R.air.lsin[m] * ci - R.air.lcos[m] * si), ch = (float)(R.air.lcos[m] * ci + R.air.lsin[m] * si);
            o[0] = (float)rx; o[1] = (float)ry; o[2] = (float)R.air.spd_post[i];
            o[3] = sh; o[4] = ch; o[5] = (float)rx; o[6] = (float)ry; o[7] = sh; o[8] = ch;
            o[9] = (float)R.air.lsp[m]; o[10] = (O == 0 || e < N + M) ? 1.0f : 2.0f;
        }
    }
}

template <int DYN, int N, int L, int O, int WPE, int MINB>
__global__ void __launch_bounds__(32 * WPE, MINB) lsm_emit_kernel(const __grid_constant__ KParams kp) {
    using ES = EmitShared<DYN, N, L, O, WPE>;
    using REC = EmitRec<DYN, N, L, O>;
    using GEO = EmitGeom<DYN, N, L, O>;
    constexpr int M = REC::M, E = REC::E, W = REC::W, EE = E * E;
    constexpr int F = GEO::F, ROWS = GEO::ROWS, CR = GEO::CR, NCHUNK = GEO::NCHUNK, NBUF = GEO::NBUF;
    constexpr int T = 32 * WPE;
    constexpr int Q = (int)(sizeof(REC) / 16);
    extern __shared__ __align__(16) unsigned char smem_raw[];
    ES& S = *reinterpret_cast<ES*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31;
    const double r2_lt = kp.r2_lt, r2_nz = kp.r2_nz;
    // the dependents (normally lsm_pair_kernel, which does not wait at its top) are released only once the agent kernel
    // this launch depends on is complete and flushed
    pdl_wait();
    pdl_launch_dependents();
    tl_start(kp.timeline, TL_EMIT_START);
    const bool masked_reset = kp.mode == MODE_RESET && kp.env_mask != nullptr;
    // compact adjacency (host-facing callers, lsm_set_compact_adjacency): ONE thresholded E x E matrix per environment +
    // the per-observer keep masks instead of the N masked copies - 1/N of the adjacency bytes cross PCIe and the host
    // expands them (lsm_expand_adjacency_host)
    const bool compact = kp.adj_base != nullptr;
    const int warp = tid >> 5;
    // fused COO edge list in process_adj order (gnn.py:376-407); the dense adjacency becomes optional
    const bool edges = kp.edge_index != nullptr;
    const bool dense = !compact && (!edges || kp.edge_dense != 0);
    if (edges && tid == 0) {
        long long b = 0;
        for (int r = 0; r < kp.edge_range; ++r) b += kp.edge_range_totals[r];
        S.range_base = b;
        if (blockIdx.x == 0 && kp.edge_range == kp.edge_num_ranges - 1)
            kp.edge_offsets[(size_t)kp.b.num_envs * N] = b + kp.edge_range_totals[kp.edge_range];     // nnz of the step
    }

    for (int k = tid; k < N * W; k += T) S.sel[k] = kp.sel_tab[k];     // visible after the first barrier of the loop below
    auto prefetch = [&](int env, int slot) {
        const int4* src = reinterpret_cast<const int4*>(kp.emit_rec + (size_t)env * sizeof(REC));
        int4* dst = reinterpret_cast<int4*>(&S.rec[slot]);
        for (int k = tid; k < Q; k += T) cp_async16(dst + k, src + k);
    };
    int it = 0, tiles = 0;
    const int env_end = kp.env_end;                 // this launch's environment range (chunked launches)
    if (kp.env_begin + (int)blockIdx.x < env_end) prefetch(kp.env_begin + blockIdx.x, 0);
    cp_async_commit();
    for (int ee = kp.env_begin + blockIdx.x; ee < env_end; ee += gridDim.x, ++it) {
        const int rb = it & 1;                         // record slot
        const int tb = NBUF == 2 ? (tiles & 1) : 0;    // tile buffer (alternates per PROCESSED environment)
        cp_async_wait_all();
        // the bulk copies that last read this iteration's tile buffers have finished reading them (bulk groups are per
        // thread: lane 0 of every warp issues a share of the copies and commits exactly one group per environment)
        if (lane == 0) { if (NBUF == 2) bulk_store_wait_read<1>(); else bulk_store_wait_read<0>(); }
        __syncthreads();
        if (ee + (int)gridDim.x < env_end) prefetch(ee + gridDim.x, rb ^ 1);
        cp_async_commit();
        // (with the fused edge list every env is re-emitted: a masked reset shifts the offsets of all later graphs)
        if (masked_reset && kp.env_mask[ee] == 0 && !edges) continue;
        ++tiles;
        const REC& R = S.rec[rb];
        float* const dthr = S.dthr[tb];
        // (a) thresholded distance matrix: d2 in float64 against the exact squared radius; the stored float32 value is
        //     d2f * rsqrt(d2f). Thread a (one per entity) walks the circular distances d = 1 .. E/2 to entity a + d
        //     (for even E the last distance only needs a < E/2), so every unordered pair is visited once.
        {
            constexpr int HALF = E / 2;                                  // circular distances 1 .. HALF
            constexpr int NSPLIT = (T / E) < 1 ? 1 : ((T / E) > HALF ? HALF : (T / E));   // threads per entity
            constexpr int DCH = (HALF + NSPLIT - 1) / NSPLIT;            // distances per thread
            for (int t = tid; t < E * NSPLIT; t += T) {
                const int part = t / E, a = t - part * E;
                const double2 pa = R.pos[a];
                if (part == 0) dthr[a * E + a] = 0.0f;
                const int d0 = part * DCH + 1;
                const int d1 = (d0 + DCH - 1) < HALF ? (d0 + DCH - 1) : HALF;
                int b = a + d0 - 1; if (b >= E) b -= E;
#pragma unroll 4
                for (int d = d0; d <= d1; ++d) {
                    b = b + 1; if (b >= E) b -= E;
                    if (E % 2 == 0 && d == HALF && a >= HALF) break;
                    const double2 pb = R.pos[b];
                    const double dx = pa.x - pb.x, dy = pa.y - pb.y;
                    const double d2 = dx * dx + dy * dy;
                    const float v = adj_value(d2, r2_lt, r2_nz);
                    dthr[a * E + b] = v; dthr[b * E + a] = v;
                }
            }
        }
        // (b) disconnected-entity bit masks before / after this step's goal updates (every warp computes the ballots,
        //     thread 0 publishes them)
        unsigned any_change = 0u, any_disc = 0u;
#pragma unroll
        for (int w = 0; w < W; ++w) {
            const int e = w * 32 + lane;
            bool dpre = false, dpost = false;
            if (e < N) { dpre = R.done[0][e] != 0; dpost = R.done[1][e] != 0; }
            else if (e < N + M) {       // obstacles (e >= N + M) are never disconnected
                const int m = e - N, order = m / N, owner = m - order * N;
                dpre = R.reached[0][owner] > order; dpost = R.reached[1][owner] > order;
            }
            const unsigned bpre = __ballot_sync(0xffffffffu, dpre), bpost = __ballot_sync(0xffffffffu, dpost);
            if (tid == 0) { S.disc[0][w] = bpre; S.disc[1][w] = bpost; }
            any_change |= (bpre ^ bpost); any_disc |= bpost;
        }
        __syncthreads();
        if (any_disc != 0u || edges) {
            for (int k = tid; k < N * W; k += T) {
                const int w = k % W;
                const unsigned sel = S.sel[k];
                S.keepm[k] = keep_word(S.disc[1][w], S.disc[0][w], sel);
            }
            __syncthreads();
        }
        if (edges) emit_edges<DYN, N, L, O, WPE>(S, kp, ee, dthr, any_change == 0u);
        if (compact) {
            unsigned* kdst = kp.adj_keep + (size_t)ee * (N * W);
            for (int k = tid; k < N * W; k += T) kdst[k] = any_disc != 0u ? S.keepm[k] : 0xffffffffu;
            if (!GEO::ADJ_BULK) {
                float* bdst = kp.adj_base + (size_t)ee * EE;
                for (int idx = tid; idx < EE; idx += T) __stcs(bdst + idx, dthr[idx]);
            }
        }
        // (d) adjacency
        float* abase = kp.b.adj + (size_t)ee * (N * EE);
        const bool adj_bulk = GEO::ADJ_BULK && any_change == 0u && dense;
        if (dense) {
            if (adj_bulk) {
                // every observer sees the same matrix: mask it once in place; thread 0 sends it N times below
                if (any_disc != 0u) {
                    for (int idx = tid; idx < EE; idx += T) {
                        const int a = idx / E, b2 = idx - a * E;
                        const bool keep = ((S.keepm[a >> 5] >> (a & 31)) & 1u) && ((S.keepm[b2 >> 5] >> (b2 & 31)) & 1u);
                        if (!keep) dthr[idx] = 0.0f;
                    }
                }
            } else if (E % 4 == 0) {
                constexpr int CPR = E / 4, CHUNKS = EE / 4;
                for (int ch = tid; ch < CHUNKS; ch += T) {
                    const int a = ch / CPR, b4 = (ch - a * CPR) * 4;
                    const float4 v = *reinterpret_cast<const float4*>(dthr + ch * 4);
                    float* dst = abase + ch * 4;
#pragma unroll
                    for (int i = 0; i < N; ++i) {
                        const bool ka = any_disc == 0u || ((S.keepm[i * W + (a >> 5)] >> (a & 31)) & 1u);
                        const unsigned nib = !ka ? 0u : (any_disc == 0u ? 0xFu : ((S.keepm[i * W + (b4 >> 5)] >> (b4 & 31)) & 0xFu));
                        float4 o;
                        o.x = (nib & 1u) ? v.x : 0.0f; o.y = (nib & 2u) ? v.y : 0.0f;
                        o.z = (nib & 4u) ? v.z : 0.0f; o.w = (nib & 8u) ? v.w : 0.0f;
                        __stcs(reinterpret_cast<float4*>(dst + i * EE), o);
                    }
                }
            } else {
                for (int idx = tid; idx < EE; idx += T) {
                    const int a = idx / E, b2 = idx - a * E;
                    const float v = dthr[idx];
#pragma unroll
                    for (int i = 0; i < N; ++i) {
                        const bool keep = any_disc == 0u ||
                                          (((S.keepm[i * W + (a >> 5)] >> (a & 31)) & 1u) &&
                                           ((S.keepm[i * W + (b2 >> 5)] >> (b2 & 31)) & 1u));
                        __stcs(abase + i * EE + idx, keep ? v : 0.0f);
                    }
                }
            }
        }
        // (c) node features: one thread per (observer, entity) row, assembled row-major in shared memory
        // graph_feat_type 'global' (navigation_graph_safe.py:1017-1036): 7-wide observer-independent rows [vel, pos, goal, type]
        const bool gfeat = (kp.c.flags & LSM_FLAG_GRAPH_FEAT_GLOBAL) != 0;
        const int Fr = gfeat ? 7 : F;
        float* nbase = kp.b.node_obs + (size_t)ee * (ROWS * Fr);
        auto node_row = [&](int r, float* o) { node_feature_row<DYN, N, L, O>(R, r, gfeat, o); };
        bool adj_sent = false;
        for (int c = 0; c < NCHUNK; ++c) {
            const int r0 = c * CR;
            const int nrows = (ROWS - r0) < CR ? (ROWS - r0) : CR;
            const int nb = NBUF == 2 ? tb : 0;
            if (c > 0) {
                // the previous chunk's copy has finished reading the buffer this chunk is written to
                if (lane == 0 && warp == WPE - 1) bulk_store_wait_read<0>();
                __syncthreads();
            }
            float* buf = S.nodes[nb];
            for (int r = tid; r < nrows; r += T) node_row(r0 + r, buf + r * Fr);
            if (GEO::NODE_BULK || adj_bulk || compact) bulk_store_fence();
            __syncthreads();
            if (lane == 0) {
                // the copies of one environment are issued by lane 0 of EVERY warp (observer i by warp i mod WPE, the node
                // chunk by the last warp) instead of by one thread while the other 127 wait at the next barrier
                const unsigned long long stream_pol = l2_evict_first();
                if (adj_bulk && !adj_sent) {
#pragma unroll 1
                    for (int i = warp; i < N; i += WPE) bulk_store(abase + i * EE, dthr, (unsigned)EE * 4u, stream_pol);
                }
                if (compact && GEO::ADJ_BULK && !adj_sent && warp == 0)
                    bulk_store(kp.adj_base + (size_t)ee * EE, dthr, (unsigned)EE * 4u, stream_pol);
                if (GEO::NODE_BULK && warp == WPE - 1) bulk_store(nbase + r0 * Fr, buf, (unsigned)(nrows * Fr) * 4u, stream_pol);
                bulk_store_commit();
            }
            adj_sent = true;
            if (!GEO::NODE_BULK) {
                const int nfl = nrows * Fr;
                if (Fr % 2 == 0 && (ROWS * Fr) % 2 == 0) {
                    for (int q = tid; q < nfl / 2; q += T)
                        __stcs(reinterpret_cast<float2*>(nbase + r0 * Fr) + q, reinterpret_cast<const float2*>(buf)[q]);
                } else {
                    for (int q = tid; q < nfl; q += T) __stcs(nbase + r0 * Fr + q, buf[q]);
                }
                __syncthreads();
            }
        }
    }
    // every bulk copy issued by this block has finished READING shared memory before the block retires
    if (lane == 0) bulk_store_wait_read<0>();
    cp_async_wait_all();
    tl_end(kp.timeline, TL_EMIT_END);
}

// ---------------------------------------------------------------------------------------------
// lsm_record_emit_kernel: graph emission from stored records (lsm_emit_from_records). One item = (record, observer i):
// observer i's node rows (E, F) and masked thresholded matrix (E, E), byte for byte what lsm_emit_kernel wrote for that
// observer, through the same three helpers. A group of WPI warps owns one item at a time (WPI grows with E so that the
// E * E stores of an item spread over more lanes); a block holds GPB groups, each synchronising on its own named barrier.
// ---------------------------------------------------------------------------------------------
// observer i's keep masks of a stored record, as lsm_emit_kernel derives them (no masking at all when nothing is
// disconnected after the step). Called by one whole warp; lanes < W write keep[lane].
template <int DYN, int N, int L, int O>
__device__ __forceinline__ void record_keep_words(const EmitRec<DYN, N, L, O>& R, const uint32_t* sel_tab, int i, int lane,
                                                  unsigned* keep) {
    using REC = EmitRec<DYN, N, L, O>;
    constexpr int M = REC::M, W = REC::W;
    unsigned pre[W], post[W], any_disc = 0u;
#pragma unroll
    for (int w = 0; w < W; ++w) {
        const int e = w * 32 + lane;
        bool dpre = false, dpost = false;
        if (e < N) { dpre = R.done[0][e] != 0; dpost = R.done[1][e] != 0; }
        else if (e < N + M) {       // obstacles (e >= N + M) are never disconnected
            const int m = e - N, order = m / N, owner = m - order * N;
            dpre = R.reached[0][owner] > order; dpost = R.reached[1][owner] > order;
        }
        pre[w] = __ballot_sync(0xffffffffu, dpre); post[w] = __ballot_sync(0xffffffffu, dpost);
        any_disc |= post[w];
    }
    if (lane < W) {
#pragma unroll
        for (int w = 0; w < W; ++w)
            if (w == lane) keep[w] = any_disc != 0u ? keep_word(post[w], pre[w], sel_tab[i * W + w]) : 0xffffffffu;
    }
}

// copy stored record `rec` into shared memory with cp.async: thread t of the TG threads of an item group; returns when
// this thread's copies have landed (the caller synchronises the group)
template <typename REC, int TG>
__device__ __forceinline__ void stage_record(REC& S, const unsigned char* records, long long rec, int t) {
    constexpr int Q = (int)(sizeof(REC) / 16);
    const int4* src = reinterpret_cast<const int4*>(records + rec * (long long)sizeof(REC));
    int4* dst = reinterpret_cast<int4*>(&S);
    for (int k = t; k < Q; k += TG) cp_async16(dst + k, src + k);
    cp_async_commit();
    cp_async_wait_all();
}

template <int DYN, int N, int L, int O>
struct RecordEmitGeom {
    using REC = EmitRec<DYN, N, L, O>;
    static constexpr int E = REC::E, W = REC::W, EE = E * E;
    static constexpr int F = DYN == LSM_DYN_DOUBLE_INTEGRATOR ? 10 : 11;
    static constexpr int WPI = E <= 32 ? 1 : E < 64 ? 2 : 4;      // warps per item
    static constexpr int GPB = 8 / WPI;                             // items in flight per 256-thread block
    static constexpr int THREADS = 32 * WPI * GPB;
    struct __align__(16) Slot {
        REC rec;
        alignas(16) float nodes[E * F];
        unsigned keep[W];
    };
    static constexpr int SMEM = (int)sizeof(Slot) * GPB;
};

template <int DYN, int N, int L, int O>
__global__ void __launch_bounds__(RecordEmitGeom<DYN, N, L, O>::THREADS) lsm_record_emit_kernel(const __grid_constant__ RecordEmitArgs a) {
    using GEO = RecordEmitGeom<DYN, N, L, O>;
    using REC = EmitRec<DYN, N, L, O>;
    constexpr int E = GEO::E, EE = GEO::EE, WPI = GEO::WPI, GPB = GEO::GPB;
    constexpr int TG = 32 * WPI;                      // threads per item
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int g = threadIdx.x / TG, t = threadIdx.x - g * TG, lane = t & 31;
    typename GEO::Slot& S = reinterpret_cast<typename GEO::Slot*>(smem_raw)[g];
    auto group_sync = [&]() {
        if (WPI == 1) __syncwarp();
        else asm volatile("bar.sync %0, %1;" :: "r"(1 + g), "r"(TG) : "memory");
    };
    const int Fr = a.gfeat ? 7 : GEO::F;
    const int NF = E * Fr;                            // node floats per item
    for (long long it = (long long)blockIdx.x * GPB + g; it < a.num_items; it += (long long)gridDim.x * GPB) {
        const long long rec = a.record[it];
        const int i = a.observer[it];
        float* const adj = a.adj != nullptr ? a.adj + it * EE : nullptr;
        float* const nob = a.node_obs != nullptr ? a.node_obs + it * NF : nullptr;
        if (rec < 0 || rec >= a.num_records || i < 0 || i >= N) {     // invalid item: zero-filled outputs
            if (adj != nullptr) for (int k = t; k < EE; k += TG) __stcs(adj + k, 0.0f);
            if (nob != nullptr) for (int k = t; k < NF; k += TG) __stcs(nob + k, 0.0f);
            continue;
        }
        group_sync();                                 // the previous item's readers of S are done
        stage_record<REC, TG>(S.rec, a.records, rec, t);
        group_sync();
        const REC& R = S.rec;
        if (t < 32) record_keep_words<DYN, N, L, O>(R, a.sel_tab, i, lane, S.keep);
        // node rows of observer i, assembled in shared memory
        if (nob != nullptr)
            for (int e = t; e < E; e += TG) node_feature_row<DYN, N, L, O>(R, i * E + e, a.gfeat != 0, S.nodes + e * Fr);
        group_sync();
        // masked thresholded matrix: every entry from the two positions (the float64 d2 is symmetric bit for bit)
        if (adj != nullptr) {
            const double r2_lt = a.r2_lt, r2_nz = a.r2_nz;
            for (int k = t; k < EE; k += TG) {
                const int ra = k / E, cb = k - ra * E;
                const double2 pa = R.pos[ra], pb = R.pos[cb];
                const double dx = pa.x - pb.x, dy = pa.y - pb.y;
                const float v = adj_value(dx * dx + dy * dy, r2_lt, r2_nz);
                const bool keep = ((S.keep[ra >> 5] >> (ra & 31)) & 1u) && ((S.keep[cb >> 5] >> (cb & 31)) & 1u);
                __stcs(adj + k, keep ? v : 0.0f);
            }
        }
        if (nob != nullptr) {
            if (NF % 4 == 0) {
                for (int k = t; k < NF / 4; k += TG) __stcs(reinterpret_cast<float4*>(nob) + k, reinterpret_cast<const float4*>(S.nodes)[k]);
            } else if (NF % 2 == 0) {
                for (int k = t; k < NF / 2; k += TG) __stcs(reinterpret_cast<float2*>(nob) + k, reinterpret_cast<const float2*>(S.nodes)[k]);
            } else {
                for (int k = t; k < NF; k += TG) __stcs(nob + k, S.nodes[k]);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// lsm_record_emit_kernel_edge_count / lsm_record_emit_kernel_edge_fill (lsm_edges_from_records): the COO edge list of
// the matrices lsm_record_emit_kernel writes for the same items, in the order of the reference's process_adj, without
// the dense matrices. Item k's edges are the non-zero entries of its masked matrix in row-major order, at node indices
// k * E + row and k * E + col. The count kernel writes counts[k], lsm_edge_scan_kernel turns the counts into offsets,
// and the fill kernel ranks each row's entries with a ballot and popcounts and writes them from offsets[k]. Same item
// groups as lsm_record_emit_kernel, same record staging and keep masks; the pattern is "adj_value != 0" and the value
// adj_value, so the edges are exactly the dense matrix's non-zeros and an edge_attr entry is bit for bit its entry.
// ---------------------------------------------------------------------------------------------
template <int DYN, int N, int L, int O>
struct RecordEdgesGeom {
    using REC = EmitRec<DYN, N, L, O>;
    static constexpr int E = REC::E, W = REC::W;
    static constexpr int WPI = RecordEmitGeom<DYN, N, L, O>::WPI;     // warps per item
    static constexpr int GPB = 8 / WPI;                                 // items in flight per 256-thread block
    static constexpr int THREADS = 32 * WPI * GPB;
    struct __align__(16) Slot {
        REC rec;
        unsigned keep[W];
        unsigned rowmask[E * W];    // fill: kept non-zero entries of every row
        int rowoff[E];              // fill: exclusive prefix of the row counts; count: the per-warp totals
    };
    static constexpr int SMEM = (int)sizeof(Slot) * GPB;
};

template <int DYN, int N, int L, int O, bool FILL>
__device__ __forceinline__ void record_edges_items(const RecordEdgesArgs& a) {
    using GEO = RecordEdgesGeom<DYN, N, L, O>;
    using REC = EmitRec<DYN, N, L, O>;
    constexpr int E = GEO::E, W = GEO::W, WPI = GEO::WPI, GPB = GEO::GPB;
    constexpr int TG = 32 * WPI;                      // threads per item
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int g = threadIdx.x / TG, t = threadIdx.x - g * TG, lane = t & 31, wg = t >> 5;
    typename GEO::Slot& S = reinterpret_cast<typename GEO::Slot*>(smem_raw)[g];
    auto group_sync = [&]() {
        if (WPI == 1) __syncwarp();
        else asm volatile("bar.sync %0, %1;" :: "r"(1 + g), "r"(TG) : "memory");
    };
    const double r2_lt = a.r2_lt, r2_nz = a.r2_nz;
    const unsigned lt = (1u << lane) - 1u;
    for (long long it = (long long)blockIdx.x * GPB + g; it < a.num_items; it += (long long)gridDim.x * GPB) {
        const long long rec = a.record[it];
        const int i = a.observer[it];
        if (rec < 0 || rec >= a.num_records || i < 0 || i >= N) {     // invalid item: no edges
            if (!FILL && t == 0) a.counts[it] = 0;
            continue;
        }
        group_sync();                                 // the previous item's readers of S are done
        stage_record<REC, TG>(S.rec, a.records, rec, t);
        group_sync();
        const REC& R = S.rec;
        if (t < 32) record_keep_words<DYN, N, L, O>(R, a.sel_tab, i, lane, S.keep);
        group_sync();
        // kept non-zero entries of every row: warp wg of the group takes rows wg, wg + WPI, ...; one ballot per 32 columns
        int cnt = 0;
        for (int ra = wg; ra < E; ra += WPI) {
            const bool ka = (S.keep[ra >> 5] >> (ra & 31)) & 1u;
            const double2 pa = R.pos[ra];
            int rc = 0;
#pragma unroll
            for (int w = 0; w < W; ++w) {
                const int cb = w * 32 + lane;
                bool nz = false;
                if (ka && cb < E) {
                    const double2 pb = R.pos[cb];
                    const double dx = pa.x - pb.x, dy = pa.y - pb.y;
                    nz = adj_value(dx * dx + dy * dy, r2_lt, r2_nz) != 0.0f;
                }
                const unsigned m = __ballot_sync(0xffffffffu, nz) & S.keep[w];
                if (FILL && lane == 0) S.rowmask[ra * W + w] = m;
                rc += __popc(m);
            }
            if (FILL) { if (lane == 0) S.rowoff[ra] = rc; }
            else cnt += rc;
        }
        if (!FILL) {
            if (WPI == 1) {
                if (lane == 0) a.counts[it] = cnt;
            } else {
                if (lane == 0) S.rowoff[wg] = cnt;
                group_sync();
                if (t == 0) {
                    int c = 0;
#pragma unroll
                    for (int w = 0; w < WPI; ++w) c += S.rowoff[w];
                    a.counts[it] = c;
                }
            }
            continue;
        }
        group_sync();
        // exclusive prefix of the row counts (the group's first warp)
        if (t < 32) {
            int running = 0;
            for (int c0 = 0; c0 < E; c0 += 32) {
                const int ra = c0 + lane;
                const int v = ra < E ? S.rowoff[ra] : 0;
                int incl = v;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += u; }
                if (ra < E) S.rowoff[ra] = running + incl - v;
                running += __shfl_sync(0xffffffffu, incl, 31);
            }
        }
        group_sync();
        // edges of row ra at offsets[it] + rowoff[ra] + rank among the row's kept non-zeros; a position outside
        // [0, capacity) (a short capacity, or offsets of other items) is never written
        const long long base = a.offsets[it], node0 = it * E;
        long long* const src = a.edge_index;
        long long* const dst = a.edge_index + a.capacity;
        const unsigned long long cap = (unsigned long long)a.capacity;
        for (int ra = wg; ra < E; ra += WPI) {
            long long p0 = base + S.rowoff[ra];
            const double2 pa = R.pos[ra];
#pragma unroll
            for (int w = 0; w < W; ++w) {
                const unsigned m = S.rowmask[ra * W + w];
                const long long p = p0 + __popc(m & lt);
                if (((m >> lane) & 1u) && (unsigned long long)p < cap) {
                    const int cb = w * 32 + lane;
                    const double2 pb = R.pos[cb];
                    const double dx = pa.x - pb.x, dy = pa.y - pb.y;
                    src[p] = node0 + ra; dst[p] = node0 + cb; a.edge_attr[p] = adj_value(dx * dx + dy * dy, r2_lt, r2_nz);
                }
                p0 += __popc(m);
            }
        }
    }
}

template <int DYN, int N, int L, int O>
__global__ void __launch_bounds__(RecordEdgesGeom<DYN, N, L, O>::THREADS)
lsm_record_emit_kernel_edge_count(const __grid_constant__ RecordEdgesArgs a) {
    record_edges_items<DYN, N, L, O, false>(a);
}

template <int DYN, int N, int L, int O>
__global__ void __launch_bounds__(RecordEdgesGeom<DYN, N, L, O>::THREADS)
lsm_record_emit_kernel_edge_fill(const __grid_constant__ RecordEdgesArgs a) {
    record_edges_items<DYN, N, L, O, true>(a);
}

}  // namespace lsm

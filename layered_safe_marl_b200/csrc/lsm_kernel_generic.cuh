// lsm_kernel_generic.cuh - step kernel with run-time N / L (any 1 <= N <= 32, N*L <= 128).
// Used for configurations that have no compile-time specialisation (lsm_kernel_spec.cuh).
#pragma once
#include "lsm_step_common.cuh"

namespace lsm {

struct EnvSmem {
    double *ax, *ay, *as2, *as3, *vpre_x, *vpre_y, *vpost_x, *vpost_y, *spd_post, *sth, *cth, *rawx, *rawy;
    double *lx, *ly, *lh, *lsp, *lsin, *lcos, *daa;
    double *ox, *oy;                    // obstacles (extension)
    float* dthr;
    int *goal_pre, *goal_post, *reached_pre, *reached_post, *done_pre, *done_post;
    unsigned *disc_pre, *disc_post, *keepm;
    __device__ __forceinline__ void bind(unsigned char* base, const SmemLayout& sl) {
        ax = (double*)(base + sl.ax); ay = (double*)(base + sl.ay); as2 = (double*)(base + sl.as2); as3 = (double*)(base + sl.as3);
        vpre_x = (double*)(base + sl.vpre_x); vpre_y = (double*)(base + sl.vpre_y);
        vpost_x = (double*)(base + sl.vpost_x); vpost_y = (double*)(base + sl.vpost_y);
        spd_post = (double*)(base + sl.spd_post); sth = (double*)(base + sl.sth); cth = (double*)(base + sl.cth);
        rawx = (double*)(base + sl.rawx); rawy = (double*)(base + sl.rawy);
        lx = (double*)(base + sl.lx); ly = (double*)(base + sl.ly); lh = (double*)(base + sl.lh);
        lsp = (double*)(base + sl.lsp); lsin = (double*)(base + sl.lsin); lcos = (double*)(base + sl.lcos);
        daa = (double*)(base + sl.daa); dthr = (float*)(base + sl.dthr);
        ox = (double*)(base + sl.ox); oy = (double*)(base + sl.oy);
        goal_pre = (int*)(base + sl.goal_pre); goal_post = (int*)(base + sl.goal_post);
        reached_pre = (int*)(base + sl.reached_pre); reached_post = (int*)(base + sl.reached_post);
        done_pre = (int*)(base + sl.done_pre); done_post = (int*)(base + sl.done_post);
        disc_pre = (unsigned*)(base + sl.disc_pre); disc_post = (unsigned*)(base + sl.disc_post);
        keepm = (unsigned*)(base + sl.keepm);
    }
};

// navigation_graph_safe.py:452-465 is_obstacle_collision (no walls): any obstacle closer than 1.05 * (size + size)
__device__ __forceinline__ bool obstacle_collision(const double* ox, const double* oy, int O, double px, double py) {
    for (int k = 0; k < O; ++k) {
        const double dx = ox[k] - px, dy = oy[k] - py;
        if (sqrt(dx * dx + dy * dy) < 1.05 * (0.050 + 0.050)) return true;
    }
    return false;
}

// World.apply_safety_filter for ONE ego agent (core.py:648-677; safety_filter.py:203-260, 378-433)
template <int DYN>
__device__ void safety_filter_agent(const KParams& kp, const Curriculum& q, const EnvSmem& S, int i, int N,
                                    double raw0, double raw1, double& safe0, double& safe1, int& filtered, int& deconf) {
    constexpr int ND = DYN == LSM_DYN_DOUBLE_INTEGRATOR ? 4 : 5;
    const lsm_config& c = kp.c;
    safe0 = raw0; safe1 = raw1; filtered = 0; deconf = -1;
    const double ex = S.ax[i], ey = S.ay[i], e2 = S.as2[i], e3 = S.as3[i];
    double best_d = 0.0, best_v = 0.0; int kd = -1, kv = -1; bool kv_in_range = false;
    for (int j = 0; j < N; ++j) {
        if (j == i || S.done_pre[j]) continue;
        const double ox = S.ax[j], oy = S.ay[j];
        const double ddx = ox - ex, ddy = oy - ey;
        const double dist = sqrt(ddx * ddx + ddy * ddy);
        double rel[ND]; bool inr;
        relative_state<DYN>(ex, ey, e2, e3, ox, oy, S.as2[j], S.as3[j], rel);
        const double v = hj_value<DYN>(kp, q, rel, inr);
        if (kd < 0 || dist < best_d) { kd = j; best_d = dist; }
        if (kv < 0 || v < best_v) { kv = j; best_v = v; kv_in_range = inr; }
    }
    if (kv < 0) return;                         // no other active agent
    deconf = kv;
    filter_resolve<DYN, false>(kp, best_d, best_v, kv_in_range, ex, ey, e2, e3, S.ax[kv], S.ay[kv], S.as2[kv], S.as3[kv],
                               raw0, raw1, S.rawx[kv], S.rawy[kv], safe0, safe1, filtered);
}

// ---------------------------------------------------------------------------------------------
// the kernel
// ---------------------------------------------------------------------------------------------
#define AFP(f) (kp.b.agent_f64 + ((size_t)(f) * (size_t)n + (size_t)env) * (size_t)N + (size_t)ai)
#define AIP(f) (kp.b.agent_i32 + ((size_t)(f) * (size_t)n + (size_t)env) * (size_t)N + (size_t)ai)
#define EFP(f) (kp.b.env_f64 + (size_t)(f) * (size_t)n + (size_t)env)
#define EIP(f) (kp.b.env_i32 + (size_t)(f) * (size_t)n + (size_t)env)

template <int DYN>
__global__ void __launch_bounds__(256) lsm_generic_kernel(const __grid_constant__ KParams kp) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const lsm_config& c = kp.c;
    const int lane = threadIdx.x & 31;
    const int warp_in_block = threadIdx.x >> 5;
    const int warps_per_block = blockDim.x >> 5;
    const int N = kp.N, L = kp.L, M = kp.M, E = kp.E, G = kp.G, EPW = kp.EPW, W = kp.W, O = kp.O;
    const int Dobs = kp.D, F = kp.F;
    const long long n = kp.b.num_envs;
    const int le = lane / G;            // local env of this lane in the per-agent phases
    const int ai = lane - le * G;       // agent index of this lane
    const unsigned group_mask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << (le * G));
    unsigned char* wbase = smem_raw + (size_t)warp_in_block * kp.smem_per_warp;
    EnvSmem S;                          // this lane's env (per-agent phases)
    S.bind(wbase + (size_t)le * kp.sl.bytes_per_env, kp.sl);
    const bool use_filter_arg = (c.flags & LSM_FLAG_USE_SAFETY_FILTER) != 0;
    const long long ngroups = (n + EPW - 1) / EPW;

    for (long long grp = (long long)blockIdx.x * warps_per_block + warp_in_block; grp < ngroups;
         grp += (long long)gridDim.x * warps_per_block) {
        const long long env0 = grp * EPW;
        const long long env = env0 + le;
        bool env_on = env < n;
        if (kp.mode == MODE_RESET && kp.env_mask != nullptr && env_on) env_on = kp.env_mask[env] != 0;
        const bool agent_on = env_on && ai < N;
        if (__ballot_sync(0xffffffffu, env_on) == 0u) continue;

        // ---------------- P0: load ----------------
        double x = 0, y = 0, s2 = 0, s3 = 0, p_dist = 0, state_time = 0, min_rel = INFINITY, goal_min_time = INFINITY;
        double times_old = -1, dists_old = -1, dist_left = -1, ep_travel_dist = 0, ep_min_dist = INFINITY, action_diff = 0;
        int reached = 0, done = 0, safety_filtered = 0, deconflict = -1, ncoll = 0;
        int ep_len = 0, ep_conflict = 0, ep_multi = 0, ep_done = 0, nobst = 0;
        int current_step = 0, reset_count = 0, parity = 0;
        double ratio = 0.0;
        if (env_on) {
            current_step = *EIP(LSM_EI_CURRENT_STEP); reset_count = *EIP(LSM_EI_RESET_COUNT);
            parity = *EIP(LSM_EI_PARITY); ratio = *EFP(LSM_EF_CURRICULUM_RATIO);
        }
        if (agent_on) {
            x = *AFP(LSM_AF_X); y = *AFP(LSM_AF_Y); s2 = *AFP(LSM_AF_S2); s3 = *AFP(LSM_AF_S3);
            p_dist = *AFP(LSM_AF_P_DIST); state_time = *AFP(LSM_AF_STATE_TIME);
            min_rel = *AFP(LSM_AF_MIN_REL_DIST); goal_min_time = *AFP(LSM_AF_GOAL_MIN_TIME);
            times_old = *AFP(parity ? LSM_AF_TIMES_REQ_B : LSM_AF_TIMES_REQ_A);
            dists_old = *AFP(parity ? LSM_AF_DISTS_GOAL_B : LSM_AF_DISTS_GOAL_A);
            dist_left = *AFP(LSM_AF_DIST_LEFT); ep_travel_dist = *AFP(LSM_AF_EP_TRAVEL_DIST);
            ep_min_dist = *AFP(LSM_AF_EP_MIN_DIST); action_diff = *AFP(LSM_AF_ACTION_DIFF);
            reached = *AIP(LSM_AI_REACHED); done = *AIP(LSM_AI_DONE);
            safety_filtered = *AIP(LSM_AI_SAFETY_FILTERED); deconflict = *AIP(LSM_AI_DECONFLICT_IDX);
            ncoll = *AIP(LSM_AI_NUM_COLLISIONS); ep_len = *AIP(LSM_AI_EP_TRAVEL_LEN);
            ep_conflict = *AIP(LSM_AI_EP_CONFLICT); ep_multi = *AIP(LSM_AI_EP_MULTI); ep_done = *AIP(LSM_AI_EP_DONE);
            if (O > 0) nobst = *AIP(LSM_AI_NUM_OBST_COLLISIONS);
        }
        double times_req = times_old, dists_goal = dists_old;
        // landmarks of the warp's EPW environments: contiguous runs per field
        {
            const long long total = (long long)EPW * M;
            for (int f = 0; f < LSM_LF_COUNT; ++f) {
                const double* src = kp.b.landmarks + ((size_t)f * (size_t)n + (size_t)env0) * (size_t)M;
                int el = 0, m = lane;
                while (m >= M) { m -= M; ++el; }
                for (long long idx = lane; idx < total; idx += 32) {
                    if (env0 + el < n) {
                        unsigned char* eb = wbase + (size_t)el * kp.sl.bytes_per_env;
                        const int off = f == 0 ? kp.sl.lx : f == 1 ? kp.sl.ly : f == 2 ? kp.sl.lh : f == 3 ? kp.sl.lsp
                                        : f == 4 ? kp.sl.lsin : kp.sl.lcos;
                        ((double*)(eb + off))[m] = src[idx];
                    }
                    m += 32;
                    while (m >= M) { m -= M; ++el; }
                }
            }
        }
        if (O > 0) {   // obstacles of the warp's environments: [2][n][O]
            for (int idx = lane; idx < EPW * O; idx += 32) {
                const int el = idx / O, k = idx - el * O;
                if (env0 + el < n) {
                    unsigned char* eb = wbase + (size_t)el * kp.sl.bytes_per_env;
                    ((double*)(eb + kp.sl.ox))[k] = kp.b.obstacles[((size_t)0 * (size_t)n + (size_t)(env0 + el)) * (size_t)O + k];
                    ((double*)(eb + kp.sl.oy))[k] = kp.b.obstacles[((size_t)1 * (size_t)n + (size_t)(env0 + el)) * (size_t)O + k];
                }
            }
        }
        Curriculum q = curriculum(kp, ratio);
        if (agent_on) {
            S.ax[ai] = x; S.ay[ai] = y; S.as2[ai] = s2; S.as3[ai] = s3;
            S.done_pre[ai] = done; S.reached_pre[ai] = reached;
        }
        __syncwarp();

        bool all_done_env = false;

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
                S.rawx[ai] = raw0; S.rawy[ai] = raw1;
            }
            __syncwarp();
            double safe0 = raw0, safe1 = raw1;
            for (int it = 0; it < c.num_internal_step; ++it) {
                if (agent_on && q.world_filter) {   // world.use_safety_filter is per env (curriculum, Q5)
                    int filt = 0, dec = -1;
                    safe0 = raw0; safe1 = raw1;
                    if (!done) safety_filter_agent<DYN>(kp, q, S, ai, N, raw0, raw1, safe0, safe1, filt, dec);
                    deconflict = dec; safety_filtered = filt;
                }
                __syncwarp();   // everyone has read the pre-integration states
                if (agent_on) {
                    const double d0 = raw0 - safe0, d1 = raw1 - safe1;
                    action_diff = sqrt(d0 * d0 + d1 * d1);
                    if (!done) integrate<DYN>(x, y, s2, s3, safe0, safe1, c.dt, p_dist, state_time);
                    S.ax[ai] = x; S.ay[ai] = y; S.as2[ai] = s2; S.as3[ai] = s3;
                }
                __syncwarp();
            }
            // ---------------- P2: agent-agent distances, goal / reward / done ----------------
            int goal_pre = 0, goal_post = 0, reached_post = reached, done_post = done;
            double rew = 0.0;
            double vpx = 0, vpy = 0, vqx = 0, vqy = 0;   // world-frame velocity pre / post own update
            double theta = 0, speed = 0;
            bool reached_now = false;
            if (agent_on) {
                // core.py:696-709 (+ the agent block of calculate_distances)
                double m = INFINITY;
                for (int j = 0; j < N; ++j) {
                    const double dx = x - S.ax[j], dy = y - S.ay[j];
                    const double d = sqrt(dx * dx + dy * dy);
                    S.daa[ai * N + j] = d;
                    if (j != ai && !done && !S.done_pre[j] && d < m) m = d;
                }
                min_rel = m;
                theta = theta_of<DYN>(s2, s3); speed = speed_of<DYN>(s2, s3);
                if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) { vpx = s2; vpy = s3; }
                else { const double ct = lsm_cos(s2), st = lsm_sin(s2); vpx = s3 * ct; vpy = s3 * st; S.cth[ai] = ct; S.sth[ai] = st; }
                goal_pre = goal_index(reached, ai, N, M);
                const double gx = S.lx[goal_pre], gy = S.ly[goal_pre], gh = S.lh[goal_pre], gs = S.lsp[goal_pre];
                // observation (pre-update goal): navigation_graph_safe.py:855-875, utils.py:114-137
                float* o = kp.b.obs + ((size_t)env * N + ai) * Dobs;
                if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) {
                    o[0] = (float)s2; o[1] = (float)s3; o[2] = (float)(gx - x); o[3] = (float)(gy - y);
                    o[4] = (float)S.lsin[goal_pre]; o[5] = (float)S.lcos[goal_pre]; o[6] = (float)gs;
                } else {
                    double rx, ry; rotate_into(gx - x, gy - y, S.cth[ai], S.sth[ai], rx, ry);
                    const double rh = gh - s2;
                    o[0] = (float)s3; o[1] = (float)rx; o[2] = (float)ry;
                    o[3] = (float)lsm_sin(rh); o[4] = (float)lsm_cos(rh); o[5] = (float)gs;
                }
                // reward_reach_goal: navigation_graph_safe.py:691-791
                const double he = direction_alignment_error(theta, gh);
                const double hpr = 1.0 - clipd(he / q.heading_thresh, 0.0, 1.0);
                const double se = fabs(speed - gs);
                const double sen = clipd(se / q.speed_thresh, 0.0, 1.0);
                double cra = ratio_sloped(ratio, 0.25, 0.75);
                if (use_filter_arg) cra = 1.0;
                reached_now = goal_reached<DYN>(x, y, theta, speed, gx, gy, gh, gs, q);
                if (reached_now) {
                    const double spr = 1.0 - sen;
                    const double pdx = gx - x, pdy = gy - y;
                    double cte = pdx * lsm_sin(theta) - pdy * lsm_cos(theta);
                    const double nrm = norm2(pdx, pdy);
                    cte = fabs(cte) / (nrm > 1e-6 ? nrm : 1e-6);
                    cte = clipd(cte, 0.0, 1.0);
                    const double pr = hpr * spr * (1.0 - cte);
                    double goal_rew;
                    if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) goal_rew = c.goal_rew * pr;
                    else goal_rew = c.goal_rew * (pr * cra + (1.0 - cra));
                    if (!done) rew += goal_rew;
                }
                if (!done) {
                    if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) {
                        if (!use_filter_arg) {   // utils.py:323-349
                            const double cg = lsm_cos(gh), sg = lsm_sin(gh);
                            double rpx, rpy, rvx, rvy;
                            rotate_into(x - gx, y - gy, cg, sg, rpx, rpy);
                            const double dist = norm2(rpx, rpy);
                            const double ang = lsm_atan2(rpy, rpx);
                            const double ang_range = kPi / 6;
                            rotate_into(s2 - 0.0, s3 - 0.0, cg, sg, rvx, rvy);
                            const double rh = magnetic_heading(rpx, rpy, 2.0 * q.dist_thresh);
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
                            hap = clipd(1.0 - q.sloped, 0.0, 1.0) * hap;
                            rew -= hap;
                        }
                        if (use_filter_arg) rew -= 1.0; else rew -= 1.0 * q.sloped;
                    } else {
                        double rpx, rpy;
                        rotate_into(x - gx, y - gy, lsm_cos(gh), lsm_sin(gh), rpx, rpy);
                        const double rs[4] = { rpx, rpy, theta - gh, speed };
                        double ttr = grid_value_rt(kp.tg, rs);
                        if (isnan(ttr)) ttr = kp.tg.ttr_max;
                        rew -= 0.04 * ttr;
                        rew -= sen * cra;
                    }
                }
                // update_reached_goal_and_done (+ freeze_agent): navigation_graph_safe.py:658-675, 1091-1099
                if (reached_now && !done) reached_post = reached + 1;
                done_post = done;
                vqx = vpx; vqy = vpy;
                if (reached_post >= L) {
                    done_post = 1;
                    if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) { s2 = 0.0; s3 = 0.0; } else s3 = 0.0;
                    vqx = 0.0; vqy = 0.0;
                    if (DYN != LSM_DYN_DOUBLE_INTEGRATOR) { vqx = s3 * S.cth[ai]; vqy = s3 * S.sth[ai]; }
                }
                goal_post = goal_index(reached_post, ai, N, M);
                S.vpre_x[ai] = vpx; S.vpre_y[ai] = vpy; S.vpost_x[ai] = vqx; S.vpost_y[ai] = vqy;
                S.spd_post[ai] = (DYN == LSM_DYN_DOUBLE_INTEGRATOR) ? 0.0 : s3;
                S.goal_pre[ai] = goal_pre; S.goal_post[ai] = goal_post;
                S.reached_post[ai] = reached_post; S.done_post[ai] = done_post;
                S.as2[ai] = s2; S.as3[ai] = s3;
            }
            __syncwarp();
            if (agent_on) {
                // remaining reward terms see agents < i after and agents > i before their own update
                if (c.flags & LSM_FLAG_SAFETY_VIOLATION) {         // navigation_graph_safe.py:793-798
                    double r = 0.0;
                    for (int a = 0; a < N; ++a) {
                        if (a == ai) continue;
                        const int adone = a < ai ? S.done_post[a] : S.done_pre[a];
                        if (S.daa[ai * N + a] < q.sep && !adone) r += q.conflict_rew;
                    }
                    rew += r;
                }
                if (c.flags & LSM_FLAG_POTENTIAL_CONFLICT) {       // navigation_graph_safe.py:800-823
                    int count = 0; double pen = 0.0;
                    for (int a = 0; a < N; ++a) {
                        if (a == ai) continue;
                        const int adone = a < ai ? S.done_post[a] : S.done_pre[a];
                        const double rd = S.daa[ai * N + a];
                        if (rd < q.eng && !adone) {
                            const double rx = S.ax[a] - x, ry = S.ay[a] - y;
                            const double closeness = 1.0 - clipd((rd - q.sep) / (q.eng - q.sep), 0.0, 1.0);
                            const double dir = lsm_atan2(ry, rx);
                            const double vax = a < ai ? S.vpost_x[a] : S.vpre_x[a];
                            const double vay = a < ai ? S.vpost_y[a] : S.vpre_y[a];
                            double change = lsm_cos(dir) * (vax - vpx) + lsm_sin(dir) * (vay - vpy);
                            change = fabs(pymin(0.0, change));
                            pen += change * closeness;
                            count += 1;
                        }
                    }
                    if (count > 1) rew += q.multi_rew * pen;
                }
                if ((c.flags & LSM_FLAG_DIFF_FROM_FILTERED_ACTION) && use_filter_arg) {   // :825-828
                    if (!done) rew += q.diff_rew * action_diff;
                }
                if (c.flags & LSM_FLAG_HJ_VALUE) {                 // :830-837, core.py:459-468
                    constexpr int ND = DYN == LSM_DYN_DOUBLE_INTEGRATOR ? 4 : 5;
                    double r = 0.0;
                    // the ego state is still the pre-update one here (reward runs before the update)
                    const double e2 = (DYN == LSM_DYN_DOUBLE_INTEGRATOR) ? vpx : theta;
                    const double e3 = (DYN == LSM_DYN_DOUBLE_INTEGRATOR) ? vpy : speed;
                    for (int a = 0; a < N; ++a) {
                        if (a == ai) continue;
                        const int adone = a < ai ? S.done_post[a] : S.done_pre[a];
                        if (adone) continue;
                        // an agent that is not done has identical pre / post state
                        double rel[ND]; bool inr;
                        double o2, o3;
                        if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) { o2 = S.vpre_x[a]; o3 = S.vpre_y[a]; }
                        else { o2 = S.as2[a]; o3 = S.as3[a]; }
                        relative_state<DYN>(x, y, e2, e3, S.ax[a], S.ay[a], o2, o3, rel);
                        const double v = hj_value<DYN>(kp, q, rel, inr);
                        const double cvp = fabs(pymin(v - 0.4, 0.0));
                        r += q.cvalue_rew * cvp;
                    }
                    rew += r;
                }
                rew = clipd(rew, c.min_reward, c.max_reward);

                // episode statistics: environment.py:1004-1022 (uses agent i's row of its own masked adj)
                if (!done_post) {
                    ep_len += 1;
                    ep_travel_dist += norm2(vqx, vqy) * c.dt;
                    int cnt = 0; bool have = false; double mn = INFINITY;
                    for (int j = 0; j < N; ++j) {
                        const int jdisc = j <= ai ? S.done_post[j] : S.done_pre[j];
                        double d = jdisc ? 0.0 : S.daa[ai * N + j];
                        d = (d < c.coordination_range && d > 0.0) ? d : 0.0;
                        if (d != 0.0) { have = true; if (d < c.engagement_distance_ref) cnt++; if (d < mn) mn = d; }
                    }
                    if (have) {
                        if (cnt > 1) ep_multi += 1;
                        if (mn < c.separation_distance_target) ep_conflict += 1;
                        if (mn < ep_min_dist) ep_min_dist = mn;
                    }
                }
                if (done_post) ep_done = 1;
                // info_callback state: navigation_graph_safe.py:386-413 (post-update goal and velocity)
                {
                    const double gx = S.lx[goal_post], gy = S.ly[goal_post];
                    const double dx = x - gx, dy = y - gy;
                    const double dist = sqrt(dx * dx + dy * dy);
                    const double th2 = theta_of<DYN>(s2, s3), sp2 = speed_of<DYN>(s2, s3);
                    const bool r2 = goal_reached<DYN>(x, y, th2, sp2, gx, gy, S.lh[goal_post], S.lsp[goal_post], q);
                    if (r2 && times_req == -1.0) { times_req = (double)current_step * c.dt; dists_goal = p_dist; dist_left = dist; }
                    if (times_req == -1.0) { dists_goal = p_dist; dist_left = dist; }
                    if (obstacle_collision(S.ox, S.oy, O, x, y)) nobst += 1;     // navigation_graph_safe.py:402-404
                    for (int a = 0; a < N; ++a) {
                        if (a == ai) continue;
                        if (S.daa[ai * N + a] < 1.05 * (0.050 + 0.050)) ncoll += 1;
                    }
                }
            }
            if (agent_on && kp.b.reward_individual != nullptr) kp.b.reward_individual[(size_t)env * N + ai] = (float)rew;
            // shared reward: sequential sum in agent order (environment.py:1032-1037)
            if (c.flags & LSM_FLAG_SHARED_REWARD) {
                double s = 0.0;
                for (int k = 0; k < N; ++k) s += __shfl_sync(0xffffffffu, rew, le * G + k);
                rew = s;
            }
            const bool done_out = done_post || (current_step >= c.episode_length);   // environment.py:260-268
            const unsigned not_done = __ballot_sync(0xffffffffu, agent_on && !done_out);
            all_done_env = env_on && ((not_done & group_mask) == 0u);
            if (agent_on) {
                kp.b.reward[(size_t)env * N + ai] = (float)rew;
                kp.b.done[(size_t)env * N + ai] = (uint8_t)done_out;
                kp.b.safe_action[((size_t)env * N + ai) * 2] = safe0;
                kp.b.safe_action[((size_t)env * N + ai) * 2 + 1] = safe1;
            }
            reached = reached_post; done = done_post;
            parity ^= 1;
        } else {
            // RESET / OBSERVE: pre == post
            if (agent_on) {
                double vx, vy;
                if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) { vx = s2; vy = s3; }
                else { const double ct = lsm_cos(s2), st = lsm_sin(s2); vx = s3 * ct; vy = s3 * st; S.cth[ai] = ct; S.sth[ai] = st; }
                const int g = goal_index(reached, ai, N, M);
                S.vpre_x[ai] = vx; S.vpre_y[ai] = vy; S.vpost_x[ai] = vx; S.vpost_y[ai] = vy;
                S.spd_post[ai] = (DYN == LSM_DYN_DOUBLE_INTEGRATOR) ? 0.0 : s3;
                S.goal_pre[ai] = g; S.goal_post[ai] = g;
                S.reached_post[ai] = reached; S.done_post[ai] = done;
            }
            __syncwarp();
        }

        // ---------------- P3: reset (graphworker auto-reset or explicit) ----------------
        const bool do_reset = (kp.mode == MODE_STEP && kp.flag && all_done_env) || (kp.mode == MODE_RESET && env_on);
        const bool sample = (kp.mode == MODE_STEP) ? true : (kp.flag != 0);
        const unsigned reset_lanes = __ballot_sync(0xffffffffu, do_reset);
        if (reset_lanes != 0u) {
            // episode summary: environment.py:895-926 (sequential sums in agent order)
            double s_len = 0, s_dist = 0, s_done = 0, s_reached = 0, s_conf = 0, s_min = 0, s_multi = 0, mn = INFINITY;
            const double len_i = ep_len == 0 ? 1.0 : (double)ep_len;
            for (int k = 0; k < N; ++k) {
                const int src = le * G + k;
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
            if (do_reset && ai == 0) {
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
            if (do_reset && kp.mode == MODE_STEP && kp.b.term_f64 != nullptr) {
                if (agent_on)
                    term_snapshot(kp.b, (size_t)env * N + ai, (size_t)kp.b.num_envs * N, x, y, min_rel, dist_left, times_req, times_old,
                                  dists_goal, dists_old, goal_min_time, ncoll, safety_filtered);
                if (agent_on && O > 0) kp.b.term_i32[(size_t)LSM_TI_NUM_OBST_COLLISIONS * (size_t)kp.b.num_envs * N + (size_t)env * N + ai] = nobst;
                if (ai == 0) kp.b.term_env_f64[env] = ratio;
            }
            if (do_reset) {
                current_step = 0;
                ratio = clipd((double)kp.episode / (double)c.num_total_episode, 0.0, 1.0);
                q = curriculum(kp, ratio);
            }
            if (do_reset && sample && ai == 0) {
                // Scenario.random_scenario: navigation_graph_safe.py:1199-1367, utils.py:39-68
                Rng r; r.init(kp.seed, (uint32_t)(kp.b.env_id_base + env), (uint32_t)reset_count);
                const double ws = c.world_size;
                double cra = ratio_sloped(ratio, 0.25, 0.75);
                if (use_filter_arg) cra = 1.0;
                // static obstacles first (:1204-1209): 0.8 * uniform(-ws/2, ws/2, 2)
                for (int k = 0; k < O; ++k) {
                    S.ox[k] = 0.8 * r.uniform(-ws / 2.0, ws / 2.0);
                    S.oy[k] = 0.8 * r.uniform(-ws / 2.0, ws / 2.0);
                }
                for (int i = 0; i < N; ++i) {
                    // :1218-1249: redraw the position while it collides with an obstacle (bounded at 1000 tries); the airtaxi
                    // speed / heading are drawn once the position is accepted
                    for (int tries = 0; tries < 1000; ++tries) {
                        if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) {
                            S.ax[i] = r.uniform(-0.8 * ws, 0.8 * ws);
                            S.ay[i] = r.uniform(-0.8 * ws, 0.8 * ws);
                        } else {
                            const double xmin = -0.5 * ws;
                            const double xmax = 0.25 * ws * cra + 0.0 * (1.0 - cra) * ws;
                            const double ry = r.uniform(-0.5 * ws, 0.5 * ws);
                            S.ax[i] = r.uniform(xmin, xmax); S.ay[i] = ry;
                        }
                        if (!obstacle_collision(S.ox, S.oy, O, S.ax[i], S.ay[i])) break;
                    }
                    if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) { S.as2[i] = 0.0; S.as3[i] = 0.0; }
                    else {
                        const double sp = r.uniform(c.goal_speed_min, c.goal_speed_max);
                        S.as2[i] = r.uniform(0.0, 2.0 * kPi);
                        S.as3[i] = sp;
                    }
                }
                for (int i = 0; i < N; ++i) {
                    // the L goals of agent i live at landmark slots l*N + i; the previous agent's at l*N + i-1
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
                                    const double d = norm2(S.lx[k * N + i] - gx, S.ly[k * N + i] - gy);
                                    if (d < dm) dm = d;
                                }
                                if (dm > min_d && dm < max_d) break;
                            }
                        } else { gx = r.uniform(xlo, xhi); gy = r.uniform(ylo, yhi); }
                        S.lx[l * N + i] = gx; S.ly[l * N + i] = gy;
                    }
                    if (i > 0) for (int l = 0; l < L; ++l) if (r.uniform(0.0, 1.0) < 0.5) {
                        S.lx[l * N + i] = S.lx[l * N + i - 1]; S.ly[l * N + i] = S.ly[l * N + i - 1];
                    }
                    if (DYN != LSM_DYN_DOUBLE_INTEGRATOR) {
                        if (S.lx[i] > S.lx[N + i]) {
                            const double tx = S.lx[i], ty = S.ly[i];
                            S.lx[i] = S.lx[N + i]; S.ly[i] = S.ly[N + i]; S.lx[N + i] = tx; S.ly[N + i] = ty;
                        }
                    }
                    for (int l = 0; l < L - 1; ++l)
                        S.lh[l * N + i] = lsm_atan2(S.ly[(l + 1) * N + i] - S.ly[l * N + i], S.lx[(l + 1) * N + i] - S.lx[l * N + i]);
                    const double last_heading = S.lh[(L - 2) * N + i];
                    const double cr = use_filter_arg ? 1.0 : ratio_sloped(ratio, 0.25, 0.75);
                    if (DYN != LSM_DYN_DOUBLE_INTEGRATOR) {
                        for (int l = 0; l < L; ++l) S.lsp[l * N + i] = c.goal_speed_max;
                    } else {
                        // goal_speeds_random is drawn before var_random; keep the draws in lsp, then decide
                        for (int l = 0; l < L; ++l) S.lsp[l * N + i] = r.uniform(c.goal_speed_min, c.goal_speed_max);
                        const double var = r.uniform(0.0, 1.0);
                        if (!(var < pymin(cr, 1.0 - 0.2))) {
                            for (int l = 0; l < L; ++l) S.lsp[l * N + i] = c.goal_speed_max;
                            S.lsp[(L - 1) * N + i] = c.goal_speed_min;
                        }
                    }
                    for (int l = 0; l < L - 1; ++l) {
                        const double pr = (DYN == LSM_DYN_DOUBLE_INTEGRATOR) ? cr * 0.25 * kPi : cra * 0.1 * kPi;
                        S.lh[l * N + i] += r.uniform(-pr, pr);
                    }
                    S.lh[(L - 1) * N + i] = last_heading;
                    for (int l = 0; l < L; ++l) {
                        S.lsin[l * N + i] = lsm_sin(S.lh[l * N + i]);
                        S.lcos[l * N + i] = lsm_cos(S.lh[l * N + i]);
                    }
                }
            }
            __syncwarp();
            if (do_reset && agent_on) {
                if (sample) { x = S.ax[ai]; y = S.ay[ai]; s2 = S.as2[ai]; s3 = S.as3[ai]; }
                done = 0; reached = 0;
                p_dist = 0.0; state_time = 0.0;
                goal_min_time = norm2(x - S.lx[ai], y - S.ly[ai]) / c.agent_max_speed;   // navigation_graph_safe.py:525-535
                times_req = -1.0; dists_goal = -1.0; dist_left = -1.0; ncoll = 0; nobst = 0;
                ep_len = 0; ep_travel_dist = 0.0; ep_done = 0; ep_conflict = 0; ep_multi = 0; ep_min_dist = INFINITY;
                double vx, vy;
                if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) { vx = s2; vy = s3; }
                else { const double ct = lsm_cos(s2), st = lsm_sin(s2); vx = s3 * ct; vy = s3 * st; S.cth[ai] = ct; S.sth[ai] = st; }
                S.ax[ai] = x; S.ay[ai] = y; S.as2[ai] = s2; S.as3[ai] = s3;
                S.vpre_x[ai] = vx; S.vpre_y[ai] = vy; S.vpost_x[ai] = vx; S.vpost_y[ai] = vy;
                S.spd_post[ai] = (DYN == LSM_DYN_DOUBLE_INTEGRATOR) ? 0.0 : s3;
                S.goal_pre[ai] = ai; S.goal_post[ai] = ai;
                S.reached_pre[ai] = 0; S.reached_post[ai] = 0; S.done_pre[ai] = 0; S.done_post[ai] = 0;
                // reset observation
                const int g = ai;
                float* o = kp.b.obs + ((size_t)env * N + ai) * Dobs;
                if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) {
                    o[0] = (float)s2; o[1] = (float)s3; o[2] = (float)(S.lx[g] - x); o[3] = (float)(S.ly[g] - y);
                    o[4] = (float)S.lsin[g]; o[5] = (float)S.lcos[g]; o[6] = (float)S.lsp[g];
                } else {
                    double rx, ry; rotate_into(S.lx[g] - x, S.ly[g] - y, S.cth[ai], S.sth[ai], rx, ry);
                    const double rh = S.lh[g] - s2;
                    o[0] = (float)s3; o[1] = (float)rx; o[2] = (float)ry;
                    o[3] = (float)lsm_sin(rh); o[4] = (float)lsm_cos(rh); o[5] = (float)S.lsp[g];
                }
            }
            if (do_reset && sample) reset_count += 1;
            __syncwarp();
            // write the new landmarks back (sampled envs only)
            if (sample) {
                for (int el = 0; el < EPW; ++el) {
                    if (!((reset_lanes >> (el * G)) & 1u)) continue;
                    unsigned char* eb = wbase + (size_t)el * kp.sl.bytes_per_env;
                    for (int f = 0; f < LSM_LF_COUNT; ++f) {
                        const int off = f == 0 ? kp.sl.lx : f == 1 ? kp.sl.ly : f == 2 ? kp.sl.lh : f == 3 ? kp.sl.lsp
                                        : f == 4 ? kp.sl.lsin : kp.sl.lcos;
                        double* dst = kp.b.landmarks + ((size_t)f * (size_t)n + (size_t)(env0 + el)) * (size_t)M;
                        for (int m = lane; m < M; m += 32) dst[m] = ((const double*)(eb + off))[m];
                    }
                    for (int k = lane; k < O; k += 32) {
                        kp.b.obstacles[((size_t)0 * (size_t)n + (size_t)(env0 + el)) * (size_t)O + k] = ((const double*)(eb + kp.sl.ox))[k];
                        kp.b.obstacles[((size_t)1 * (size_t)n + (size_t)(env0 + el)) * (size_t)O + k] = ((const double*)(eb + kp.sl.oy))[k];
                    }
                }
            }
        } else if (kp.mode == MODE_OBSERVE && agent_on) {
            // observation of the injected state
            const int g = S.goal_pre[ai];
            float* o = kp.b.obs + ((size_t)env * N + ai) * Dobs;
            if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) {
                o[0] = (float)s2; o[1] = (float)s3; o[2] = (float)(S.lx[g] - x); o[3] = (float)(S.ly[g] - y);
                o[4] = (float)S.lsin[g]; o[5] = (float)S.lcos[g]; o[6] = (float)S.lsp[g];
            } else {
                double rx, ry; rotate_into(S.lx[g] - x, S.ly[g] - y, S.cth[ai], S.sth[ai], rx, ry);
                const double rh = S.lh[g] - s2;
                o[0] = (float)s3; o[1] = (float)rx; o[2] = (float)ry;
                o[3] = (float)lsm_sin(rh); o[4] = (float)lsm_cos(rh); o[5] = (float)S.lsp[g];
            }
        }

        // ---------------- state write-back ----------------
        if (kp.mode != MODE_OBSERVE) {
            if (env_on && ai == 0) {
                *EIP(LSM_EI_CURRENT_STEP) = current_step; *EIP(LSM_EI_RESET_COUNT) = reset_count;
                *EIP(LSM_EI_PARITY) = parity; *EIP(LSM_EI_JUST_RESET) = do_reset ? 1 : 0;
                *EFP(LSM_EF_CURRICULUM_RATIO) = ratio;
            }
            if (agent_on) {
                *AFP(LSM_AF_X) = x; *AFP(LSM_AF_Y) = y; *AFP(LSM_AF_S2) = s2; *AFP(LSM_AF_S3) = s3;
                *AFP(LSM_AF_P_DIST) = p_dist; *AFP(LSM_AF_STATE_TIME) = state_time;
                *AFP(LSM_AF_MIN_REL_DIST) = min_rel; *AFP(LSM_AF_GOAL_MIN_TIME) = goal_min_time;
                // the slot named by `parity` receives the newest values; the other keeps last step's
                *AFP(parity ? LSM_AF_TIMES_REQ_B : LSM_AF_TIMES_REQ_A) = times_req;
                *AFP(parity ? LSM_AF_DISTS_GOAL_B : LSM_AF_DISTS_GOAL_A) = dists_goal;
                if (do_reset) {
                    *AFP(parity ? LSM_AF_TIMES_REQ_A : LSM_AF_TIMES_REQ_B) = times_req;
                    *AFP(parity ? LSM_AF_DISTS_GOAL_A : LSM_AF_DISTS_GOAL_B) = dists_goal;
                }
                *AFP(LSM_AF_DIST_LEFT) = dist_left; *AFP(LSM_AF_EP_TRAVEL_DIST) = ep_travel_dist;
                *AFP(LSM_AF_EP_MIN_DIST) = ep_min_dist; *AFP(LSM_AF_ACTION_DIFF) = action_diff;
                *AIP(LSM_AI_REACHED) = reached; *AIP(LSM_AI_DONE) = done;
                *AIP(LSM_AI_SAFETY_FILTERED) = safety_filtered; *AIP(LSM_AI_DECONFLICT_IDX) = deconflict;
                *AIP(LSM_AI_NUM_COLLISIONS) = ncoll; *AIP(LSM_AI_EP_TRAVEL_LEN) = ep_len;
                *AIP(LSM_AI_EP_CONFLICT) = ep_conflict; *AIP(LSM_AI_EP_MULTI) = ep_multi; *AIP(LSM_AI_EP_DONE) = ep_done;
                if (O > 0) *AIP(LSM_AI_NUM_OBST_COLLISIONS) = nobst;
            }
        }
        __syncwarp();

        // ---------------- P4: graph observation for the warp's environments ----------------
        for (int el = 0; el < EPW; ++el) {
            const long long ee = env0 + el;
            if (ee >= n) break;
            if (kp.mode == MODE_RESET && kp.env_mask != nullptr && kp.env_mask[ee] == 0) continue;
            EnvSmem T;
            T.bind(wbase + (size_t)el * kp.sl.bytes_per_env, kp.sl);
            // (a) pairwise distances, thresholded by the sensing radius (core.py:514-543 and the strict
            //     0 < d < R test of navigation_graph_safe.py:991)
            for (int e = lane; e < E; e += 32) T.dthr[e * E + e] = 0.0f;
            for (int p = lane; p < kp.num_pairs; p += 32) {
                const int a = kp.pair_tab[2 * p], b2 = kp.pair_tab[2 * p + 1];
                // entity order agents, landmarks, obstacles (core.py:489-496)
                const double pax = a < N ? T.ax[a] : (a < N + M ? T.lx[a - N] : T.ox[a - N - M]);
                const double pay = a < N ? T.ay[a] : (a < N + M ? T.ly[a - N] : T.oy[a - N - M]);
                const double pbx = b2 < N ? T.ax[b2] : (b2 < N + M ? T.lx[b2 - N] : T.ox[b2 - N - M]);
                const double pby = b2 < N ? T.ay[b2] : (b2 < N + M ? T.ly[b2 - N] : T.oy[b2 - N - M]);
                const double dx = pax - pbx, dy = pay - pby;
                const double d = sqrt(dx * dx + dy * dy);
                const float v = (d < c.coordination_range && d > 0.0) ? (float)d : 0.0f;
                T.dthr[a * E + b2] = v; T.dthr[b2 * E + a] = v;
            }
            // (b) disconnected-entity bit masks, before and after this step's goal updates
            unsigned any_disc = 0u;
            for (int w = 0; w < W; ++w) {
                const int e = w * 32 + lane;
                bool dpre = false, dpost = false;
                if (e < N) { dpre = T.done_pre[e] != 0; dpost = T.done_post[e] != 0; }
                else if (e < N + M) {   // obstacles (e >= N + M) are never disconnected
                    const int m = e - N, owner = m % N, order = m / N;
                    dpre = T.reached_pre[owner] > order; dpost = T.reached_post[owner] > order;
                }
                const unsigned bpre = __ballot_sync(0xffffffffu, dpre), bpost = __ballot_sync(0xffffffffu, dpost);
                if (lane == 0) { T.disc_pre[w] = bpre; T.disc_post[w] = bpost; }
                any_disc |= bpost;
            }
            __syncwarp();
            // keep mask of observer i: entities owned by agents <= i are seen post-update, the others pre-update
            for (int k = lane; k < N * W; k += 32) {
                const int w = k % W;
                const unsigned sel = kp.sel_tab[k];
                T.keepm[k] = ~((T.disc_post[w] & sel) | (T.disc_pre[w] & ~sel));
            }
            __syncwarp();
            // (c) node features: one lane per (observer, entity) row
            {
                float* nbase = kp.b.node_obs + (size_t)ee * N * E * F;
                const int rows = N * E;
                int i = 0, e = lane;
                while (e >= E) { e -= E; ++i; }
                for (int r = lane; r < rows; r += 32) {
                    float* o = nbase + (size_t)r * F;
                    const double xi = T.ax[i], yi = T.ay[i];
                    const double vix = T.vpost_x[i], viy = T.vpost_y[i];
                    if (kp.c.flags & LSM_FLAG_GRAPH_FEAT_GLOBAL) {
                        // _get_entity_feat_global (navigation_graph_safe.py:1017-1036): [vel, pos, goal_pos, type]; an agent's
                        // goal is its FIRST landmark (optimal_match_index = arange, :179), a landmark's goal is itself
                        if (e < N) {
                            const bool post = e <= i;
                            o[0] = (float)(post ? T.vpost_x[e] : T.vpre_x[e]); o[1] = (float)(post ? T.vpost_y[e] : T.vpre_y[e]);
                            o[2] = (float)T.ax[e]; o[3] = (float)T.ay[e];
                            o[4] = (float)T.lx[e]; o[5] = (float)T.ly[e]; o[6] = 0.0f;
                        } else if (e < N + M) {
                            const int m = e - N;
                            o[0] = 0.0f; o[1] = 0.0f; o[2] = (float)T.lx[m]; o[3] = (float)T.ly[m];
                            o[4] = o[2]; o[5] = o[3]; o[6] = 1.0f;
                        } else {   // obstacle: velocity 0, goal = own position, type 2 (:1030-1032)
                            const int k = e - N - M;
                            o[0] = 0.0f; o[1] = 0.0f; o[2] = (float)T.ox[k]; o[3] = (float)T.oy[k];
                            o[4] = o[2]; o[5] = o[3]; o[6] = 2.0f;
                        }
                    } else if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) {
                        float f0, f1, f2, f3, f4, f5, f6, f7, f8, f9;
                        if (e < N) {
                            const bool post = e <= i;
                            const int g = post ? T.goal_post[e] : T.goal_pre[e];
                            const double vex = post ? T.vpost_x[e] : T.vpre_x[e], vey = post ? T.vpost_y[e] : T.vpre_y[e];
                            f0 = (float)(T.ax[e] - xi); f1 = (float)(T.ay[e] - yi);
                            f2 = (float)(vex - vix); f3 = (float)(vey - viy);
                            f4 = (float)(T.lx[g] - xi); f5 = (float)(T.ly[g] - yi);
                            f6 = (float)T.lsin[g]; f7 = (float)T.lcos[g]; f8 = (float)T.lsp[g]; f9 = 0.0f;
                        } else if (e < N + M) {
                            const int m = e - N;
                            f0 = (float)(T.lx[m] - xi); f1 = (float)(T.ly[m] - yi);
                            f2 = (float)(-vix); f3 = (float)(-viy); f4 = f0; f5 = f1;
                            f6 = (float)T.lsin[m]; f7 = (float)T.lcos[m]; f8 = (float)T.lsp[m]; f9 = 1.0f;
                        } else {   // obstacle (extension): the landmark row with heading 0, speed 0; type 2
                            const int k = e - N - M;
                            f0 = (float)(T.ox[k] - xi); f1 = (float)(T.oy[k] - yi);
                            f2 = (float)(-vix); f3 = (float)(-viy); f4 = f0; f5 = f1;
                            f6 = 0.0f; f7 = 1.0f; f8 = 0.0f; f9 = 2.0f;
                        }
                        float2* o2 = reinterpret_cast<float2*>(o);   // rows are 40 B: 8 B aligned
                        o2[0] = make_float2(f0, f1); o2[1] = make_float2(f2, f3); o2[2] = make_float2(f4, f5);
                        o2[3] = make_float2(f6, f7); o2[4] = make_float2(f8, f9);
                    } else {
                        const double ci = T.cth[i], si = T.sth[i];
                        if (e < N) {
                            const bool post = e <= i;
                            const int g = post ? T.goal_post[e] : T.goal_pre[e];
                            const double vex = post ? T.vpost_x[e] : T.vpre_x[e], vey = post ? T.vpost_y[e] : T.vpre_y[e];
                            double rx, ry, gx, gy;
                            rotate_into(T.ax[e] - xi, T.ay[e] - yi, ci, si, rx, ry);
                            rotate_into(T.lx[g] - xi, T.ly[g] - yi, ci, si, gx, gy);
                            // sin/cos(theta_e - theta_i) and sin/cos(goal_heading - theta_i) by angle difference
                            const double ce = T.cth[e], se = T.sth[e];
                            o[0] = (float)rx; o[1] = (float)ry; o[2] = (float)norm2(vex - vix, vey - viy);
                            o[3] = (float)(se * ci - ce * si); o[4] = (float)(ce * ci + se * si);
                            o[5] = (float)gx; o[6] = (float)gy;
                            o[7] = (float)(T.lsin[g] * ci - T.lcos[g] * si); o[8] = (float)(T.lcos[g] * ci + T.lsin[g] * si);
                            o[9] = (float)T.lsp[g]; o[10] = 0.0f;
                        } else {
                            // landmark, or obstacle (extension): the landmark row with heading 0 (sin 0, cos 1), speed 0; type 2
                            const int m = e - N;
                            const bool is_obst = e >= N + M;
                            const double px = is_obst ? T.ox[m - M] : T.lx[m], py = is_obst ? T.oy[m - M] : T.ly[m];
                            const double ls = is_obst ? 0.0 : T.lsin[m], lc = is_obst ? 1.0 : T.lcos[m];
                            double rx, ry;
                            rotate_into(px - xi, py - yi, ci, si, rx, ry);
                            const float sh = (float)(ls * ci - lc * si), ch = (float)(lc * ci + ls * si);
                            o[0] = (float)rx; o[1] = (float)ry; o[2] = (float)T.spd_post[i];
                            o[3] = sh; o[4] = ch; o[5] = (float)rx; o[6] = (float)ry; o[7] = sh; o[8] = ch;
                            o[9] = is_obst ? 0.0f : (float)T.lsp[m]; o[10] = is_obst ? 2.0f : 1.0f;
                        }
                    }
                    e += 32;
                    while (e >= E) { e -= E; ++i; }
                }
            }
            // (d) adjacency: observer i keeps entity k unless it is disconnected as seen after agents <= i updated
            {
                float* abase = kp.b.adj + (size_t)ee * N * E * E;
                const int EE = E * E;
                if (kp.adj_vec == 4) {
                    const int chunks = EE / 4, cpr = E / 4;
                    for (int ch = lane; ch < chunks; ch += 32) {
                        const int a = ch / cpr, b4 = (ch - a * cpr) * 4;
                        const float4 v = *reinterpret_cast<const float4*>(T.dthr + a * E + b4);
                        float* dst = abase + a * E + b4;
                        if (any_disc == 0u) {
                            for (int i = 0; i < N; ++i) *reinterpret_cast<float4*>(dst + (size_t)i * EE) = v;
                        } else {
                            for (int i = 0; i < N; ++i) {
                                const bool ka = (T.keepm[i * W + (a >> 5)] >> (a & 31)) & 1u;
                                const unsigned nib = ka ? ((T.keepm[i * W + (b4 >> 5)] >> (b4 & 31)) & 0xFu) : 0u;
                                float4 o;
                                o.x = (nib & 1u) ? v.x : 0.0f; o.y = (nib & 2u) ? v.y : 0.0f;
                                o.z = (nib & 4u) ? v.z : 0.0f; o.w = (nib & 8u) ? v.w : 0.0f;
                                *reinterpret_cast<float4*>(dst + (size_t)i * EE) = o;
                            }
                        }
                    }
                } else {
                    for (int idx = lane; idx < EE; idx += 32) {
                        const int a = idx / E, b2 = idx - a * E;
                        const float v = T.dthr[idx];
                        for (int i = 0; i < N; ++i) {
                            const bool keep = ((T.keepm[i * W + (a >> 5)] >> (a & 31)) & 1u) &&
                                              ((T.keepm[i * W + (b2 >> 5)] >> (b2 & 31)) & 1u);
                            abase[(size_t)i * EE + idx] = keep ? v : 0.0f;
                        }
                    }
                }
            }
            __syncwarp();
        }
        __syncwarp();
    }
}

}  // namespace lsm

// lsm_step_common.cuh - device functions shared by the generic and the specialised step kernels.
#pragma once
#include "lsm_grid.cuh"

namespace lsm {

__constant__ double c_mag_cos[kMagSegments];
__constant__ double c_mag_sin[kMagSegments];

// utils.py:276-321, with cos/sin(phi_k) tabulated by the host
__device__ double magnetic_heading(double px, double py, double radius) {
    if (fabs(px) < 1e-6) return 0.0;
    const double scale_x = 0.5;
    px = scale_x * px;
    double bx = 0.0, by = 0.0;
    for (int k = 0; k < kMagSegments; ++k) {
        const double c = c_mag_cos[k], s = c_mag_sin[k];
        const double Ly = -radius * c, Lz = -radius * s;
        const double dLy = radius * s, dLz = -radius * c;
        const double rx = px - 0.0, ry = py - Ly, rz = 0.0 - Lz;
        const double rmag = sqrt((rx * rx + ry * ry) + rz * rz);
        const double rmag3 = rmag * rmag * rmag;
        const double cx = dLy * rz - dLz * ry;
        const double cy = dLz * rx - 0.0 * rz;
        bx = bx + cx / rmag3;
        by = by + cy / rmag3;
    }
    bx = bx / scale_x;
    return lsm_atan2(by, bx);
}

__device__ __forceinline__ int goal_index(int reached, int i, int N, int M) {   // navigation_graph_safe.py:576-582
    int order = reached * N + i;
    if (order >= M) order = (reached - 1) * N + i;
    return order;
}

// relative state between ego and other (safety_filter.py:277-284, 356-362)
template <int DYN>
__device__ __forceinline__ void relative_state(double ex, double ey, double e2, double e3, double ox, double oy,
                                               double o2, double o3, double (&r)[DYN == LSM_DYN_DOUBLE_INTEGRATOR ? 4 : 5]) {
    if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) {
        r[0] = ex - ox; r[1] = ey - oy; r[2] = e2 - o2; r[3] = e3 - o3;
    } else {
        const double ddx = ox - ex, ddy = oy - ey;
        const double dist = sqrt(ddx * ddx + ddy * ddy);
        const double ang = lsm_atan2(ddy, ddx);
        double sa, ca;
        lsm_sincos(ang - e2, &sa, &ca);          // exactly lsm_cos / lsm_sin of the same argument, one reduction
        r[0] = dist * ca;
        r[1] = dist * sa;
        r[2] = o2 - e2; r[3] = e3; r[4] = o3;
    }
}

// The same relative state with the airtaxi position written as a rotation into the ego frame:
//   d cos(phi - theta_e) = dx cos(theta_e) + dy sin(theta_e),  d sin(phi - theta_e) = dy cos(theta_e) - dx sin(theta_e)
// (phi = atan2(dy, dx), d = |(dx, dy)|) - equal to safety_filter.py:277-284 to ~1e-16 d, one sincos instead of
// sqrt + atan2 + cos + sin per pair. Used by the specialised pipeline; the generic kernel keeps the literal form.
// (se, ce) = lsm_sincos(e2), passed in by callers that already have them (airtaxi only; ignored for the double integrator)
template <int DYN>
__device__ __forceinline__ void relative_state_rot_sc(double ex, double ey, double e2, double e3, double ox, double oy,
                                                      double o2, double o3, double se, double ce,
                                                      double (&r)[DYN == LSM_DYN_DOUBLE_INTEGRATOR ? 4 : 5]) {
    if constexpr (DYN == LSM_DYN_DOUBLE_INTEGRATOR) {
        r[0] = ex - ox; r[1] = ey - oy; r[2] = e2 - o2; r[3] = e3 - o3;
    } else {
        const double ddx = ox - ex, ddy = oy - ey;
        r[0] = ddx * ce + ddy * se;
        r[1] = ddy * ce - ddx * se;
        r[2] = o2 - e2; r[3] = e3; r[4] = o3;
    }
}
template <int DYN>
__device__ __forceinline__ void relative_state_rot(double ex, double ey, double e2, double e3, double ox, double oy,
                                                   double o2, double o3, double (&r)[DYN == LSM_DYN_DOUBLE_INTEGRATOR ? 4 : 5]) {
    double se = 0.0, ce = 1.0;
    if constexpr (DYN != LSM_DYN_DOUBLE_INTEGRATOR) lsm_sincos(e2, &se, &ce);
    relative_state_rot_sc<DYN>(ex, ey, e2, e3, ox, oy, o2, o3, se, ce, r);
}

// HJ value of the generic kernel (safety_filter.py:192-201, 345-354); out of range (in_range = false, +inf) for a NaN
// position or a NaN value
template <int DYN>
__device__ __forceinline__ double hj_value(const KParams& kp, const Curriculum& q,
                                           const double (&rel)[DYN == LSM_DYN_DOUBLE_INTEGRATOR ? 4 : 5], bool& in_range) {
    const double v = grid_value_rt(kp.vg, rel);
    in_range = !isnan(v);
    if (!in_range) return INFINITY;
    return v - (q.sep - kp.vg.separation_distance);
}

// Second half of the safety handles (safety_filter.py:225-260, 400-433) once the deconflicting agent
// `kv` (first minimum of the HJ value) and the smallest distance are known: gradient lookup,
// least-restrictive bang-bang or CBF-QP, control clipping, filtered flag.
// SPEC: the specialised pipeline and the operator - relative state in the rotation form (relative_state_rot_sc, with
// (se, ce) = lsm_sincos(e2) of the caller), gradient inline in the arithmetic F32. Otherwise the generic kernel - the
// literal relative_state, gradient in the handle's arithmetic chosen at run time (grid_grad_rt).
template <int DYN, bool SPEC, bool F32 = false>
__device__ __forceinline__ void filter_resolve(const KParams& kp, double best_d, double best_v, bool kv_in_range,
                                               double ex, double ey, double e2, double e3,
                                               double ox, double oy, double o2, double o3,
                                               double raw0, double raw1, double oraw0, double oraw1,
                                               double& safe0, double& safe1, int& filtered,
                                               double se = 0.0, double ce = 1.0) {
    constexpr int ND = DYN == LSM_DYN_DOUBLE_INTEGRATOR ? 4 : 5;
    const lsm_config& c = kp.c;
    if (best_d > c.coordination_range) return;
    if (!kv_in_range) return;
    double rel[ND];
    double g[ND];
    if constexpr (SPEC) {
        relative_state_rot_sc<DYN>(ex, ey, e2, e3, ox, oy, o2, o3, se, ce, rel);
        grid_grad<ND, F32>(kp.vg, rel, g);
    } else {
        relative_state<DYN>(ex, ey, e2, e3, ox, oy, o2, o3, rel);
        grid_grad_rt(kp.vg, rel, g);
    }
    const double uref[4] = { raw0, raw1, oraw0, oraw1 };
    const double eps_hj = 0.4;
    double u[4]; bool aliased = false;
    const double dt = c.dt;
    if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) {
        const double a[4] = { g[2], g[3], -g[2], -g[3] };
        if (best_v < eps_hj) {
#pragma unroll
            for (int k = 0; k < 4; ++k) u[k] = (a[k] < 0.0) ? -0.5 : 0.5;
        } else {
            double b = g[0] * rel[2] + g[1] * rel[3];
            b = b + c.cbf_rate * best_v;
            const double pinv[4] = { 1.0, 1.0, 1.0, 1.0 };
            if (!qp_project(a, b, uref, pinv, u)) {
                aliased = true;
#pragma unroll
                for (int k = 0; k < 4; ++k) u[k] = uref[k];
            }
        }
        const double axmax = (rel[2] < 0.5 - dt * 0.5) ? 0.5 : 0.0;
        const double axmin = (rel[2] > -0.5 - dt * (-0.5)) ? -0.5 : 0.0;
        u[0] = pymax(pymin(u[0], axmax), axmin);
        const double aymax = (rel[3] < 0.5 - dt * 0.5) ? 0.5 : 0.0;
        const double aymin = (rel[3] > -0.5 - dt * (-0.5)) ? -0.5 : 0.0;
        u[1] = pymax(pymin(u[1], aymax), aymin);
    } else {
        const double wmax = 0.1, amin = -0.001, amax = 0.002;
        const double vmin = 60 * 0.514444 * 0.001, vmax = 175 * 0.514444 * 0.001;
        double a[4];
        a[0] = (g[0] * rel[1] + g[1] * (-rel[0])) + g[2] * (-1.0);
        a[1] = g[2]; a[2] = g[3]; a[3] = g[ND - 1];
        const bool bang = best_v < eps_hj;
        if (bang) {
            double lo[4] = { f32r(-wmax), f32r(-wmax), f32r(amin), f32r(amin) };
            double hi[4] = { f32r(wmax), f32r(wmax), f32r(amax), f32r(amax) };
            // cascade of whole-vector jnp.where selections (safety_filter.py:70-78): the LAST true one wins
            int which = 0;
            if (rel[3] <= vmin) which = 1;
            if (rel[3] >= vmax) which = 2;
            if (rel[ND - 1] <= vmin) which = 3;
            if (rel[ND - 1] >= vmax) which = 4;
            if (which == 1) lo[2] = 0.0;
            if (which == 2) hi[2] = 0.0;
            if (which == 3) lo[3] = 0.0;
            if (which == 4) hi[3] = 0.0;
#pragma unroll
            for (int k = 0; k < 4; ++k) u[k] = (a[k] < 0.0) ? lo[k] : hi[k];
        } else {
            double s2r, c2r;
            lsm_sincos(rel[2], &s2r, &c2r);
            const double f0 = -rel[3] + rel[ND - 1] * c2r;
            const double f1 = rel[ND - 1] * s2r;
            double b = g[0] * f0 + g[1] * f1;
            b = b + c.cbf_rate * best_v;
            double pinv[4];
            if (rel[0] < 0.0) { pinv[0] = 1.0 / 100.0; pinv[1] = 1.0 / 10.0; pinv[2] = 1.0 / 10.0; pinv[3] = 1.0 / 1.0; }
            else { pinv[0] = 1.0 / 10.0; pinv[1] = 1.0 / 1.0; pinv[2] = 1.0 / 100.0; pinv[3] = 1.0 / 10.0; }
            if (!qp_project(a, b, uref, pinv, u)) {
                aliased = true;
#pragma unroll
                for (int k = 0; k < 4; ++k) u[k] = uref[k];
            } else {
                u[0] = pymax(pymin(u[0], wmax), -wmax);
                u[2] = pymax(pymin(u[2], wmax), -wmax);
            }
        }
        double cmax = (rel[3] < vmax - dt * amax) ? amax : 0.0;
        double cmin = (rel[3] > vmin - dt * amin) ? amin : 0.0;
        u[1] = pymax(pymin(u[1], cmax), cmin);
        cmax = (rel[ND - 1] < vmax - dt * amax) ? amax : 0.0;
        cmin = (rel[ND - 1] > vmin - dt * amin) ? amin : 0.0;
        u[3] = pymax(pymin(u[3], cmax), cmin);
        if (bang) { u[1] = f32r(u[1]); u[3] = f32r(u[3]); }
    }
    double nd = 0.0;
    if (!aliased) {
#pragma unroll
        for (int k = 0; k < 4; ++k) { const double d = u[k] - uref[k]; nd = nd + d * d; }
        nd = sqrt(nd);
    }
    filtered = nd > 1e-4;
    safe0 = u[0]; safe1 = u[1];
}

// Terminal-step snapshot of what info_callback reads (navigation_graph_safe.py:386-450) for an environment that is
// about to auto-reset: graphworker returns the terminal step's infos (env_wrappers.py:861-874), the reset below would
// overwrite them.
__device__ __forceinline__ void term_snapshot(const lsm_buffers& b, size_t a, size_t fstride, double x, double y, double min_rel,
                                              double dist_left, double times_new, double times_old, double dists_new,
                                              double dists_old, double goal_min_time, int ncoll, int safety_filtered) {
    double* tf = b.term_f64 + a;
    tf[LSM_TF_X * fstride] = x; tf[LSM_TF_Y * fstride] = y; tf[LSM_TF_MIN_REL_DIST * fstride] = min_rel;
    tf[LSM_TF_DIST_LEFT * fstride] = dist_left; tf[LSM_TF_TIMES_REQ_NEW * fstride] = times_new;
    tf[LSM_TF_TIMES_REQ_OLD * fstride] = times_old; tf[LSM_TF_DISTS_GOAL_NEW * fstride] = dists_new;
    tf[LSM_TF_DISTS_GOAL_OLD * fstride] = dists_old; tf[LSM_TF_GOAL_MIN_TIME * fstride] = goal_min_time;
    int* ti = b.term_i32 + a;
    ti[LSM_TI_NUM_COLLISIONS * fstride] = ncoll; ti[LSM_TI_SAFETY_FILTERED * fstride] = safety_filtered;
}

// core.py:191-210 / :110-131, closed-form over one dt
// airtaxi, `sc` != nullptr: sc[0..1] = lsm_sincos(theta before the step) from the caller; on return sc[0..1] =
// lsm_sincos(theta after the step) - the per-agent kernel needs both anyway (filter frame before, velocity after).
template <int DYN>
__device__ __forceinline__ void integrate(double& x, double& y, double& s2, double& s3, double u0, double u1, double dt,
                                          double& p_dist, double& state_time, double* sc = nullptr) {
    if (DYN == LSM_DYN_DOUBLE_INTEGRATOR) {
        double vx = s2, vy = s3;
        x = x + vx * dt + 0.5 * u0 * dt * dt;
        y = y + vy * dt + 0.5 * u1 * dt * dt;
        vx = vx + u0 * dt; vy = vy + u1 * dt;
        double speed = sqrt(vx * vx + vy * vy);
        const double max_speed = 0.5;
        if (speed > max_speed) { vx = max_speed * vx / speed; vy = max_speed * vy / speed; }
        s2 = vx; s3 = vy;
        speed = sqrt(vx * vx + vy * vy);
        p_dist += speed * dt;
    } else {
        const double vmin = 60 * 0.514444 * 0.001, vmax = 175 * 0.514444 * 0.001;
        const double th0 = s2, v0 = s3, om = u0, ac = u1;
        const double th1 = th0 + om * dt;
        double v1 = v0 + ac * dt;
        double ddx, ddy;
        double s0, c0, s1 = 0.0, c1 = 1.0;
        if (sc != nullptr) { s0 = sc[0]; c0 = sc[1]; } else lsm_sincos(th0, &s0, &c0);
        const bool small = fabs(om * dt) < 1e-3;
        if (sc != nullptr || !small) lsm_sincos(th1, &s1, &c1);
        if (sc != nullptr) { sc[0] = s1; sc[1] = c1; }
        if (small) {
            const double T = dt, o = om;
            const double i0 = T, i1 = T * T / 2.0, i2 = T * T * T / 3.0, i3 = T * T * T * T / 4.0, i4 = T * T * T * T * T / 5.0;
            const double cc0 = c0, cc1 = -s0 * o, cc2 = -c0 * o * o / 2.0, cc3 = s0 * o * o * o / 6.0;
            const double sc0 = s0, sc1 = c0 * o, sc2 = -s0 * o * o / 2.0, sc3 = -c0 * o * o * o / 6.0;
            ddx = v0 * (cc0 * i0 + cc1 * i1 + cc2 * i2 + cc3 * i3) + ac * (cc0 * i1 + cc1 * i2 + cc2 * i3 + cc3 * i4);
            ddy = v0 * (sc0 * i0 + sc1 * i1 + sc2 * i2 + sc3 * i3) + ac * (sc0 * i1 + sc1 * i2 + sc2 * i3 + sc3 * i4);
        } else {
            ddx = (v1 * s1 - v0 * s0) / om + ac * (c1 - c0) / (om * om);
            ddy = (-(v1 * c1) + v0 * c0) / om + ac * (s1 - s0) / (om * om);
        }
        x = x + ddx; y = y + ddy;
        s2 = th1;
        if (v1 > vmax) v1 = vmax;
        if (v1 < vmin) v1 = vmin;
        s3 = v1;
        p_dist += v1 * dt;
    }
    state_time += dt;
}

}  // namespace lsm

/*
 * lsm_b200_hj.h - C ABI of the HJ reachability solver (liblsm_b200_hj.so): computes the backward reachable tube value
 * function that the safety filter consumes, for the relative double-integrator and airtaxi dynamics of the filter
 * (oracle/lsm_oracle.c apply_safety_filter). Nothing here needs an environment handle, so the solver lives in its own
 * library, next to the simulator's liblsm_b200.so.
 *
 * Plain pointers and sizes only. `initial`, `out` and `work` are DEVICE pointers owned by the caller; `horizons` is a
 * HOST array. All launches and copies go to the cudaStream_t passed as `stream` (void*; NULL = default), on the caller's
 * current device. No entry point synchronises. Every function that can fail returns 0 on success, a non-zero code
 * otherwise, and then lsm_hj_last_error() describes the failure (thread-local string): 2 = invalid arguments,
 * 100 + cudaError_t = a launch or copy failed.
 *
 * The scheme (DESIGN.md "HJ value functions"; tests/hj_solve_oracle.py restates it op for op), in float64 throughout:
 *   lattice      node k of dim d at lo[d] + k * spacing[d]; spacing = (hi-lo)/n on periodic dims, (hi-lo)/(n-1)
 *                otherwise; values C-order, last dim fastest. Double integrator [px, py, vx, vy] (no periodic dim),
 *                airtaxi [x_r, y_r, theta_rel (periodic), v_a, v_b].
 *   derivatives  WENO5 (Jiang-Peng) left / right derivatives from v[k-3 .. k+3] per dim; ghosts wrap on periodic dims
 *                and extrapolate away from zero on the others.
 *   Hamiltonian  H(x, p) = p . f(x) + sum_k a_k u*_k, a = p^T G, with the filter's drift, control Jacobian,
 *                float32-rounded boxes and airtaxi speed saturation. The controls split into the ego's and the other
 *                agent's: double integrator [ax_e, ay_e | ax_o, ay_o] (k = 0, 1 | 2, 3), airtaxi [w_a, w_b, a_a, a_b]
 *                with k = 0, 2 the ego's and k = 1, 3 the other's. The ego's controls maximise, u*_k = a_k < 0 ? lo_k :
 *                hi_k. The other agent's depend on the game:
 *                  0 cooperative  maximise as well (lsm_hj_solve; no disturbance);
 *                  1 adversarial  minimise, u*_k = a_k < 0 ? hi_k : lo_k (a disturbance, disturbance_mode 'min');
 *                  2 constant     held at 0: their terms are dropped from H (the other keeps its velocity, or its
 *                                 turn rate and speed).
 *   dissipation  global Lax-Friedrichs: dV/dtau = min(0, H(x, (p- + p+)/2) + sum_i alpha_i (p+_i - p-_i)/2), alpha
 *                from the lattice (lsm_hj_dissipation, lsm_hj_game_dissipation): alpha_i = max |f_i| + sum_k max |G_ik|
 *                max(|lo_k|, |hi_k|) over the controls in play. Cooperative and adversarial: [max|vx|, max|vy|, 1, 1]
 *                and [f0 + W max|y|, f1 + W max|x|, 2 W, A, A]; constant: [max|vx|, max|vy|, 0.5, 0.5] and
 *                [f0 + W max|y|, f1 + W max|x|, W, A, 0], with f0 = max |-v_a + v_b cos theta|, f1 = max |v_b sin theta|
 *                over the nodes, W = 0.1 and A = max(|a_min|, |a_max|) = 0.002 (float32-rounded).
 *   time         tau from 0; steps of dt = cfl / sum_i(alpha_i / spacing_i), the last one before each horizon clipped
 *                to land on it; Shu-Osher TVD-RK3.
 *
 * The airtaxi time-to-reach grid (DESIGN.md "Time-to-reach grid"; tests/hj_ttr_oracle.py restates it op for op) is the
 * same scheme on a reach problem, also declared:
 *   state        [x, y, theta (periodic), v]: one airtaxi relative to its goal, position rotated into the goal's frame,
 *                heading minus the goal's heading, speed (the point the airtaxi reward looks up).
 *   Hamiltonian  x' = v cos theta, y' = v sin theta, theta' = w, v' = a; the controls MINIMISE:
 *                H = p0 v cos theta + p1 v sin theta + sum_k a_k (a_k < 0 ? hi_k : lo_k), a = (p2, p3), with the value
 *                function solve's float32-rounded boxes w in +-0.1, a in [-0.001, 0.002] and its speed saturation
 *                (v <= V_MIN: a >= 0; v >= V_MAX: a <= 0; each test restarting from the unsaturated box).
 *                dV/dtau = min(0, H + sum_i alpha_i (p+_i - p-_i)/2) as above.
 *   dissipation  alpha = [max |v cos theta|, max |v sin theta|, 0.1, 0.002] over the nodes.
 *   arrival      ttr = 0 where target <= 0. Elsewhere the first RK3 step whose end value V1 is <= 0 writes
 *                tau0 + h * (V0 / (V0 - V1)), with tau0, V0 the step's start and h its length; a cell is written once.
 *                Cells not reached by the horizon stay +inf.
 */
#ifndef LSM_B200_HJ_H
#define LSM_B200_HJ_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LSM_HJ_ABI_VERSION 1

int lsm_hj_abi_version(void);
const char *lsm_hj_last_error(void);

typedef struct lsm_hj_problem {
    int32_t dynamics;               /* 0 = double integrator (4-D), 1 = airtaxi (5-D) */
    int32_t shape[5];               /* nodes per dim, each >= 2; entries past the dynamics' ndim are ignored */
    double lo[5];                   /* finite, lo < hi */
    double hi[5];
    double cfl;                     /* 0 < cfl <= 1 (0.75 is hj_reachability's default) */
} lsm_hj_problem;

/* Bytes of the `work` buffer lsm_hj_solve needs: three stage arrays of cells doubles, the coordinate vectors and the
 * cos / sin table of the theta nodes (uploaded by lsm_hj_solve). 0 when the problem is invalid. */
int64_t lsm_hj_work_bytes(const lsm_hj_problem *problem);

/* Host only: the Lax-Friedrichs coefficients alpha[ndim] (entries past ndim set to 0) and the CFL time step. */
int lsm_hj_dissipation(const lsm_hj_problem *problem, double alpha[5], double *dt);

/* Solve from V(0) = initial (cells doubles) to each horizon in `horizons` (host, K finite values >= 0, non-decreasing)
 * and write V(horizons[k]) to out + k * cells. A horizon of 0 gives `initial`; a repeated horizon gives the same array
 * again. `work`: lsm_hj_work_bytes bytes, 8-byte aligned; `initial` and `out` must not overlap it. */
int lsm_hj_solve(const lsm_hj_problem *problem, const double *initial, const double *horizons, int32_t K, double *out,
                 void *work, void *stream);

/* lsm_hj_dissipation and lsm_hj_solve for a game: 0 cooperative, 1 adversarial, 2 constant (the Hamiltonian above);
 * any other value is refused with code 2. Game 0 is lsm_hj_dissipation / lsm_hj_solve bit for bit. The same work
 * buffer (lsm_hj_work_bytes), arguments and stream rules as those. */
int lsm_hj_game_dissipation(const lsm_hj_problem *problem, int32_t game, double alpha[5], double *dt);
int lsm_hj_game_solve(const lsm_hj_problem *problem, int32_t game, const double *initial, const double *horizons,
                      int32_t K, double *out, void *work, void *stream);

typedef struct lsm_hj_ttr_problem {
    int32_t shape[4];               /* nodes per dim [x, y, theta, v], each >= 2; theta is periodic */
    double lo[4];                   /* finite, lo < hi */
    double hi[4];
    double cfl;                     /* 0 < cfl <= 1 */
} lsm_hj_ttr_problem;

/* Bytes of the `work` buffer of the time-to-reach solve: three stage arrays of cells doubles, the coordinate vectors
 * and the cos / sin table of the theta nodes. 0 when the problem is invalid. */
int64_t lsm_hj_ttr_work_bytes(const lsm_hj_ttr_problem *problem);

/* Host only: the time-to-reach solve's Lax-Friedrichs coefficients alpha[4] and its CFL time step. */
int lsm_hj_ttr_dissipation(const lsm_hj_ttr_problem *problem, double alpha[4], double *dt);

/* Solve the reach problem of `target` (cells doubles, <= 0 on the target) to `horizon` (host, finite, >= 0) and write
 * the first-arrival times to `ttr` (cells doubles; +inf where not reached) and, unless NULL, V(horizon) to
 * `final_values`. `work`: the work-bytes size above, 8-byte aligned, overlapping none of the other arrays; `ttr` may
 * alias `target`. */
int lsm_hj_ttr_solve(const lsm_hj_ttr_problem *problem, const double *target, double horizon, double *ttr,
                     double *final_values, void *work, void *stream);

#ifdef __cplusplus
}
#endif
#endif

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
 *   Hamiltonian  H(x, p) = p . f(x) + sum_k a_k u*_k, a = p^T G, u*_k = a_k < 0 ? lo_k : hi_k (both agents' controls
 *                maximise, no disturbance), with the filter's drift, control Jacobian, float32-rounded boxes and airtaxi
 *                speed saturation.
 *   dissipation  global Lax-Friedrichs: dV/dtau = min(0, H(x, (p- + p+)/2) + sum_i alpha_i (p+_i - p-_i)/2), alpha
 *                from the lattice (lsm_hj_dissipation).
 *   time         tau from 0; steps of dt = cfl / sum_i(alpha_i / spacing_i), the last one before each horizon clipped
 *                to land on it; Shu-Osher TVD-RK3.
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

#ifdef __cplusplus
}
#endif
#endif

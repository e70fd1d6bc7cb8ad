// lsm_hj.cu - the HJ reachability solver declared in include/lsm_b200_hj.h (liblsm_b200_hj.so).
//
// lsm_hj_stage_kernel<DYN, STAGE, GAME>: one thread per lattice cell and one launch per TVD-RK3 stage. A thread reads
// the 7-point window of the stage input along every dim (ghost nodes built in registers), forms the WENO5 left / right
// derivatives, the global Lax-Friedrichs Hamiltonian of the game (the other agent's controls maximise, minimise or are
// held at 0; the ego's maximise) and min(0, .), and writes the stage's RK combination
// c0 * u0 + c1 * (u + h * L(u)). Stage 3 writes in place over u0: a cell reads u0 only at itself, so three stage arrays
// suffice. The window loads of a warp are 32 consecutive cells at one offset, so every load is coalesced; the reuse
// between neighbouring cells is served by L1 / L2 (the default grids are 6-26 MB).
//
// lsm_hj_ttr_stage_kernel<STAGE>: the same stencil for the airtaxi time-to-reach solve, 4-D [x, y, theta (periodic),
// v] in the goal's frame, with the controls minimising (a reach problem). Its stage 3 holds V0 = u0[cell] and V1, the
// step's end value, in registers and writes the first-arrival time of a cell whose V has just crossed to <= 0:
// tau0 + h * (V0 / (V0 - V1)), once (the slot stays +inf until then). lsm_hj_ttr_init_kernel sets the slot to 0 on
// the target (l <= 0) and +inf elsewhere. The TTR kernels have their own template and parameters so that the value
// function kernels above compile exactly as before.
//
// Every float64 operation is written out in the order of tests/hj_solve_oracle.py (tests/hj_ttr_oracle.py for the TTR
// solve), and the library is built with -fmad=false, so the solve is bit for bit the numpy restatement.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/lsm_b200_hj.h"
#include "../../include/lsm_math.h"

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) { g_err = msg; return code; }
int cuda_fail(cudaError_t e, const std::string& what) {
    g_err = what + ": " + cudaGetErrorString(e);
    return 100 + (int)e;
}

constexpr int BLOCK = 256;
constexpr double C13 = 1.0 / 3.0, C16 = 1.0 / 6.0, C56 = 5.0 / 6.0, C76 = 7.0 / 6.0, C116 = 11.0 / 6.0;
constexpr double C1312 = 13.0 / 12.0, C23 = 2.0 / 3.0, WENO_EPS = 1e-6;

// control boxes of the safety filter (HjDataHandle, Air4dCooperativeDynamics): float32-rounded, as JAX stores them
constexpr double DI_U = 0.5;
constexpr double AT_W = (double)(float)0.1, AT_AMIN = (double)(float)-0.001, AT_AMAX = (double)(float)0.002;
constexpr double AT_VMIN = 60 * 0.514444 * 0.001, AT_VMAX = 175 * 0.514444 * 0.001;

template <int DYN> struct Dims { static constexpr int ND = DYN == 0 ? 4 : 5; static constexpr int PERIODIC = DYN == 0 ? -1 : 2; };

struct StageParams {
    const double* u;                // stencil input (u0, u1 or u2)
    const double* u0;               // the step's start, read at the cell itself (stages 2 and 3)
    double* out;
    const double* coords;           // concatenated coordinate vectors
    const double* cth;              // cos / sin of the theta nodes (airtaxi)
    const double* sth;
    int64_t cells;
    int64_t n[5], stride[5], coord_off[5];
    double inv_dx[5], alpha[5];
    double h;
};

__device__ __forceinline__ double sgn(double x) { return x > 0.0 ? 1.0 : (x < 0.0 ? -1.0 : 0.0); }

// Jiang-Peng WENO5 from the five one-sided differences (Osher-Fedkiw 3.4)
__device__ __forceinline__ double weno5(double v1, double v2, double v3, double v4, double v5) {
    const double phi1 = (v1 * C13 - v2 * C76) + v3 * C116;
    const double phi2 = (v2 * -C16 + v3 * C56) + v4 * C13;
    const double phi3 = (v3 * C13 + v4 * C56) - v5 * C16;
    double a = (v1 - 2.0 * v2) + v3, b = (v1 - 4.0 * v2) + 3.0 * v3;
    const double s1 = C1312 * (a * a) + 0.25 * (b * b);
    a = (v2 - 2.0 * v3) + v4; b = v2 - v4;
    const double s2 = C1312 * (a * a) + 0.25 * (b * b);
    a = (v3 - 2.0 * v4) + v5; b = (3.0 * v3 - 4.0 * v4) + v5;
    const double s3 = C1312 * (a * a) + 0.25 * (b * b);
    const double t1 = s1 + WENO_EPS, t2 = s2 + WENO_EPS, t3 = s3 + WENO_EPS;
    const double a1 = 0.1 / (t1 * t1), a2 = 0.6 / (t2 * t2), a3 = 0.3 / (t3 * t3);
    return ((a1 * phi1 + a2 * phi2) + a3 * phi3) / ((a1 + a2) + a3);
}

// the window v[k-3 .. k+3] of dim d around `cell` (index k): wrapped on the periodic dim, ghosts extrapolated away from
// zero on the others; -> left and right derivatives
template <bool PERIODIC>
__device__ __forceinline__ void derivs(const double* __restrict__ u, int64_t cell, int64_t k, int64_t n, int64_t s,
                                       double inv_dx, double& left, double& right) {
    double w[7];
#pragma unroll
    for (int j = 0; j < 7; ++j) {
        int64_t i = k - 3 + j;
        if (PERIODIC) {
            if (i < 0) i += n;
            if (i < 0) i += n;
            if (i >= n) i -= n;
            if (i >= n) i -= n;
        } else {
            i = i < 0 ? 0 : (i > n - 1 ? n - 1 : i);
        }
        w[j] = __ldg(u + cell + (i - k) * s);
    }
    if (!PERIODIC) {
        if (k < 3) {
            const double v0 = __ldg(u + cell - k * s), v1 = __ldg(u + cell + (1 - k) * s);
            const double g = sgn(v0) * fabs(v1 - v0);
#pragma unroll
            for (int j = 0; j < 3; ++j)
                if (k - 3 + j < 0) w[j] = v0 + g * (double)(3 - k - j);
        }
        if (k > n - 4) {
            const double vn = __ldg(u + cell + (n - 1 - k) * s), vm = __ldg(u + cell + (n - 2 - k) * s);
            const double g = sgn(vn) * fabs(vn - vm);
#pragma unroll
            for (int j = 4; j < 7; ++j)
                if (k - 3 + j > n - 1) w[j] = vn + g * (double)(k - 3 + j - (n - 1));
        }
    }
    double D[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) D[j] = (w[j + 1] - w[j]) * inv_dx;
    left = weno5(D[0], D[1], D[2], D[3], D[4]);
    right = weno5(D[5], D[4], D[3], D[2], D[1]);
}

// The games (include/lsm_b200_hj.h lsm_hj_game_solve): what the other agent's controls do in H
enum Game { COOPERATIVE = 0, ADVERSARIAL = 1, CONSTANT = 2 };

// H's term of control k with switching function a and box [lo, hi]: the ego's controls (double integrator k = 0, 1;
// airtaxi k = 0, 2) maximise; the other agent's maximise (cooperative), minimise (adversarial) or are held at 0
// (constant: no term)
template <int DYN, int GAME>
__device__ __forceinline__ double control_term(double H, int k, double a, double lo, double hi) {
    const bool other = DYN == 0 ? k >= 2 : (k & 1) != 0;
    if (GAME == COOPERATIVE || !other) return H + a * (a < 0.0 ? lo : hi);
    if (GAME == ADVERSARIAL) return H + a * (a < 0.0 ? hi : lo);
    return H;
}

// STAGE 0: u + h L(u);  1: 3/4 u0 + 1/4 (u + h L(u));  2: 1/3 u0 + 2/3 (u + h L(u)). GAME is the last template
// parameter, so the cooperative instantiations are the kernel lsm_hj_solve always ran, with GAME = 0 added to the name.
template <int DYN, int STAGE, int GAME>
__global__ void __launch_bounds__(BLOCK) lsm_hj_stage_kernel(const StageParams p) {
    constexpr int ND = Dims<DYN>::ND;
    const int64_t cell = (int64_t)blockIdx.x * BLOCK + threadIdx.x;
    if (cell >= p.cells) return;
    int64_t idx[ND];
    int64_t r = cell;
#pragma unroll
    for (int d = ND - 1; d >= 0; --d) { idx[d] = r % p.n[d]; r /= p.n[d]; }
    double pl[ND], pr[ND];
#pragma unroll
    for (int d = 0; d < ND; ++d) {
        if (d == Dims<DYN>::PERIODIC) derivs<true>(p.u, cell, idx[d], p.n[d], p.stride[d], p.inv_dx[d], pl[d], pr[d]);
        else derivs<false>(p.u, cell, idx[d], p.n[d], p.stride[d], p.inv_dx[d], pl[d], pr[d]);
    }
    double q[ND];
#pragma unroll
    for (int d = 0; d < ND; ++d) q[d] = (pl[d] + pr[d]) * 0.5;
    double H;
    if (DYN == 0) {
        const double vx = p.coords[p.coord_off[2] + idx[2]], vy = p.coords[p.coord_off[3] + idx[3]];
        H = q[0] * vx + q[1] * vy;
        const double a[4] = {q[2], q[3], -q[2], -q[3]};
#pragma unroll
        for (int k = 0; k < 4; ++k) H = control_term<DYN, GAME>(H, k, a[k], -DI_U, DI_U);
    } else {
        const double x = p.coords[p.coord_off[0] + idx[0]], y = p.coords[p.coord_off[1] + idx[1]];
        const double c = p.cth[idx[2]], s = p.sth[idx[2]];
        const double va = p.coords[p.coord_off[3] + idx[3]], vb = p.coords[p.coord_off[4] + idx[4]];
        const double f0 = -va + vb * c, f1 = vb * s;
        H = q[0] * f0 + q[1] * f1;
        const double a[4] = {(q[0] * y + q[1] * (-x)) + q[2] * (-1.0), q[2], q[3], q[4]};
        // Air4dCooperativeDynamics.optimal_control_and_disturbance: each test starts from the unsaturated boxes
        double lo2 = AT_AMIN, hi2 = AT_AMAX, lo3 = AT_AMIN, hi3 = AT_AMAX;
        if (va <= AT_VMIN) { lo2 = AT_AMIN; hi2 = AT_AMAX; lo3 = AT_AMIN; hi3 = AT_AMAX; lo2 = 0.0; }
        if (va >= AT_VMAX) { lo2 = AT_AMIN; hi2 = AT_AMAX; lo3 = AT_AMIN; hi3 = AT_AMAX; hi2 = 0.0; }
        if (vb <= AT_VMIN) { lo2 = AT_AMIN; hi2 = AT_AMAX; lo3 = AT_AMIN; hi3 = AT_AMAX; lo3 = 0.0; }
        if (vb >= AT_VMAX) { lo2 = AT_AMIN; hi2 = AT_AMAX; lo3 = AT_AMIN; hi3 = AT_AMAX; hi3 = 0.0; }
        const double lo[4] = {-AT_W, -AT_W, lo2, lo3}, hi[4] = {AT_W, AT_W, hi2, hi3};
#pragma unroll
        for (int k = 0; k < 4; ++k) H = control_term<DYN, GAME>(H, k, a[k], lo[k], hi[k]);
    }
    double diss = p.alpha[0] * ((pr[0] - pl[0]) * 0.5);
#pragma unroll
    for (int d = 1; d < ND; ++d) diss = diss + p.alpha[d] * ((pr[d] - pl[d]) * 0.5);
    const double hh = H + diss;
    const double L = hh < 0.0 ? hh : 0.0;
    const double next = __ldg(p.u + cell) + p.h * L;
    double v;
    if (STAGE == 0) v = next;
    else if (STAGE == 1) v = 0.75 * p.u0[cell] + 0.25 * next;
    else v = C13 * p.u0[cell] + C23 * next;
    p.out[cell] = v;
}

// the time-to-reach solve (include/lsm_b200_hj.h lsm_hj_ttr_problem): 4-D, dim 2 periodic
struct TtrParams {
    const double* u;                // stencil input (u0, u1 or u2)
    const double* u0;               // the step's start, read at the cell itself (stages 2 and 3)
    double* out;
    double* ttr;                    // first-arrival times, +inf until the cell is reached
    const double* coords;           // concatenated coordinate vectors
    const double* cth;              // cos / sin of the theta nodes
    const double* sth;
    int64_t cells;
    int64_t n[4], stride[4], coord_off[4];
    double inv_dx[4], alpha[4];
    double h, tau0;                 // the step's length and start
};

constexpr double UNREACHED = (double)INFINITY;

__global__ void __launch_bounds__(BLOCK) lsm_hj_ttr_init_kernel(const double* __restrict__ l, double* __restrict__ ttr,
                                                                int64_t cells) {
    const int64_t cell = (int64_t)blockIdx.x * BLOCK + threadIdx.x;
    if (cell < cells) ttr[cell] = l[cell] <= 0.0 ? 0.0 : UNREACHED;
}

// STAGE as lsm_hj_stage_kernel; x' = v cos th, y' = v sin th, th' = w, v' = a with both controls minimising
template <int STAGE>
__global__ void __launch_bounds__(BLOCK) lsm_hj_ttr_stage_kernel(const TtrParams p) {
    const int64_t cell = (int64_t)blockIdx.x * BLOCK + threadIdx.x;
    if (cell >= p.cells) return;
    int64_t idx[4];
    int64_t r = cell;
#pragma unroll
    for (int d = 3; d >= 0; --d) { idx[d] = r % p.n[d]; r /= p.n[d]; }
    double pl[4], pr[4];
#pragma unroll
    for (int d = 0; d < 4; ++d) {
        if (d == 2) derivs<true>(p.u, cell, idx[d], p.n[d], p.stride[d], p.inv_dx[d], pl[d], pr[d]);
        else derivs<false>(p.u, cell, idx[d], p.n[d], p.stride[d], p.inv_dx[d], pl[d], pr[d]);
    }
    double q[4];
#pragma unroll
    for (int d = 0; d < 4; ++d) q[d] = (pl[d] + pr[d]) * 0.5;
    const double c = p.cth[idx[2]], s = p.sth[idx[2]];
    const double v = p.coords[p.coord_off[3] + idx[3]];
    const double f0 = v * c, f1 = v * s;
    double H = q[0] * f0 + q[1] * f1;
    // the filter solver's speed saturation: each test starts from the unsaturated box
    double lo3 = AT_AMIN, hi3 = AT_AMAX;
    if (v <= AT_VMIN) { lo3 = AT_AMIN; hi3 = AT_AMAX; lo3 = 0.0; }
    if (v >= AT_VMAX) { lo3 = AT_AMIN; hi3 = AT_AMAX; hi3 = 0.0; }
    const double a[2] = {q[2], q[3]}, lo[2] = {-AT_W, lo3}, hi[2] = {AT_W, hi3};
#pragma unroll
    for (int k = 0; k < 2; ++k) H = H + a[k] * (a[k] < 0.0 ? hi[k] : lo[k]);
    double diss = p.alpha[0] * ((pr[0] - pl[0]) * 0.5);
#pragma unroll
    for (int d = 1; d < 4; ++d) diss = diss + p.alpha[d] * ((pr[d] - pl[d]) * 0.5);
    const double hh = H + diss;
    const double L = hh < 0.0 ? hh : 0.0;
    const double next = __ldg(p.u + cell) + p.h * L;
    if (STAGE == 0) p.out[cell] = next;
    else if (STAGE == 1) p.out[cell] = 0.75 * p.u0[cell] + 0.25 * next;
    else {
        const double v0 = p.u0[cell];
        const double v1 = C13 * v0 + C23 * next;
        p.out[cell] = v1;
        // a cell with a time has V <= 0 at a step end; every other one has V0 > 0, so V0 - V1 > 0
        if (v1 <= 0.0 && p.ttr[cell] == UNREACHED) p.ttr[cell] = p.tau0 + p.h * (v0 / (v0 - v1));
    }
}

template <int DYN, int GAME>
cudaError_t launch_step(StageParams p, double* u0, double* u1, double* u2, double h, cudaStream_t st) {
    const unsigned grid = (unsigned)((p.cells + BLOCK - 1) / BLOCK);
    p.h = h;
    p.u = u0; p.u0 = u0; p.out = u1;
    lsm_hj_stage_kernel<DYN, 0, GAME><<<grid, BLOCK, 0, st>>>(p);
    p.u = u1; p.out = u2;
    lsm_hj_stage_kernel<DYN, 1, GAME><<<grid, BLOCK, 0, st>>>(p);
    p.u = u2; p.out = u0;
    lsm_hj_stage_kernel<DYN, 2, GAME><<<grid, BLOCK, 0, st>>>(p);
    return cudaGetLastError();
}

template <int GAME>
cudaError_t launch_game_step(int dyn, const StageParams& p, double* u0, double* u1, double* u2, double h,
                             cudaStream_t st) {
    return dyn == 0 ? launch_step<0, GAME>(p, u0, u1, u2, h, st) : launch_step<1, GAME>(p, u0, u1, u2, h, st);
}

cudaError_t launch_ttr_step(TtrParams p, double* u0, double* u1, double* u2, double tau0, double h, cudaStream_t st) {
    const unsigned grid = (unsigned)((p.cells + BLOCK - 1) / BLOCK);
    p.h = h;
    p.tau0 = tau0;
    p.u = u0; p.u0 = u0; p.out = u1;
    lsm_hj_ttr_stage_kernel<0><<<grid, BLOCK, 0, st>>>(p);
    p.u = u1; p.out = u2;
    lsm_hj_ttr_stage_kernel<1><<<grid, BLOCK, 0, st>>>(p);
    p.u = u2; p.out = u0;
    lsm_hj_ttr_stage_kernel<2><<<grid, BLOCK, 0, st>>>(p);
    return cudaGetLastError();
}

constexpr int64_t MAX_CELLS = (int64_t)1 << 38;      // keeps the launch grid within 2^31 - 1 blocks

struct Lattice {
    int nd = 0;
    int64_t cells = 0;
    double sp[5] = {0, 0, 0, 0, 0};
    std::vector<double> coords;     // concatenated per dim
    int64_t off[5] = {0, 0, 0, 0, 0};
    std::vector<double> cth, sth;   // cos / sin of the periodic dim's (theta's) nodes
};

// -> 0 and the lattice of nd dims (`periodic`: the periodic dim, -1 for none), or 2 with the message in g_err
int build_lattice(int nd, int periodic, const int32_t* shape, const double* lo_, const double* hi_, double cfl,
                  const std::string& fn, Lattice& L) {
    if (!(cfl > 0.0 && cfl <= 1.0)) return fail(2, fn + ": cfl must be in (0, 1]");
    L.nd = nd;
    L.cells = 1;
    for (int d = 0; d < L.nd; ++d) {
        const double lo = lo_[d], hi = hi_[d];
        if (shape[d] < 2) return fail(2, fn + ": every dim needs at least 2 nodes");
        if (!(std::isfinite(lo) && std::isfinite(hi) && lo < hi)) return fail(2, fn + ": every dim needs finite lo < hi");
        L.cells *= shape[d];
        if (L.cells > MAX_CELLS) return fail(2, fn + ": grid too large");
        L.sp[d] = d == periodic ? (hi - lo) / (double)shape[d] : (hi - lo) / (double)(shape[d] - 1);
    }
    for (int d = 0; d < L.nd; ++d) {
        L.off[d] = (int64_t)L.coords.size();
        for (int k = 0; k < shape[d]; ++k) L.coords.push_back(lo_[d] + L.sp[d] * (double)k);
    }
    if (periodic >= 0)
        for (int k = 0; k < shape[periodic]; ++k) {
            const double th = L.coords[L.off[periodic] + k];
            L.cth.push_back(lsm_cos(th));
            L.sth.push_back(lsm_sin(th));
        }
    return 0;
}

int check_problem(const lsm_hj_problem* pr, const char* fn, Lattice& L) {
    if (!pr) return fail(2, std::string(fn) + ": problem is NULL");
    if (pr->dynamics != 0 && pr->dynamics != 1)
        return fail(2, std::string(fn) + ": dynamics must be 0 (double integrator) or 1 (airtaxi)");
    return build_lattice(pr->dynamics == 0 ? 4 : 5, pr->dynamics == 0 ? -1 : 2, pr->shape, pr->lo, pr->hi, pr->cfl, fn,
                         L);
}

int check_ttr_problem(const lsm_hj_ttr_problem* pr, const char* fn, Lattice& L) {
    if (!pr) return fail(2, std::string(fn) + ": problem is NULL");
    return build_lattice(4, 2, pr->shape, pr->lo, pr->hi, pr->cfl, fn, L);
}

double max_abs(const double* v, int n) {
    double m = 0.0;
    for (int k = 0; k < n; ++k) m = fmax(m, fabs(v[k]));
    return m;
}

double cfl_step(const Lattice& L, const double* alpha, double cfl) {
    double s = alpha[0] / L.sp[0];
    for (int d = 1; d < L.nd; ++d) s = s + alpha[d] / L.sp[d];
    return cfl / s;
}

// alpha_i = max |f_i| + sum_k max |G_ik| max(|lo_k|, |hi_k|) over the controls in play: all four (cooperative,
// adversarial) or the ego's two (constant)
void dissipation(const lsm_hj_problem* pr, int game, const Lattice& L, double alpha[5], double* dt) {
    for (int d = 0; d < 5; ++d) alpha[d] = 0.0;
    const double* c = L.coords.data();
    if (pr->dynamics == 0) {
        alpha[0] = max_abs(c + L.off[2], pr->shape[2]);
        alpha[1] = max_abs(c + L.off[3], pr->shape[3]);
        alpha[2] = game == CONSTANT ? DI_U : DI_U + DI_U;
        alpha[3] = game == CONSTANT ? DI_U : DI_U + DI_U;
    } else {
        double f0 = 0.0, f1 = 0.0;
        for (int t = 0; t < pr->shape[2]; ++t)
            for (int a = 0; a < pr->shape[3]; ++a)
                for (int b = 0; b < pr->shape[4]; ++b) {
                    const double va = c[L.off[3] + a], vb = c[L.off[4] + b];
                    f0 = fmax(f0, fabs(-va + vb * L.cth[t]));
                    f1 = fmax(f1, fabs(vb * L.sth[t]));
                }
        alpha[0] = f0 + AT_W * max_abs(c + L.off[1], pr->shape[1]);
        alpha[1] = f1 + AT_W * max_abs(c + L.off[0], pr->shape[0]);
        alpha[2] = game == CONSTANT ? AT_W : AT_W + AT_W;
        alpha[3] = fmax(fabs(AT_AMIN), fabs(AT_AMAX));
        alpha[4] = game == CONSTANT ? 0.0 : alpha[3];
    }
    *dt = cfl_step(L, alpha, pr->cfl);
}

// TTR: alpha = [max |v cos th|, max |v sin th|, W, max(|a_min|, |a_max|)] over the nodes
void ttr_dissipation(const lsm_hj_ttr_problem* pr, const Lattice& L, double alpha[4], double* dt) {
    const double* c = L.coords.data();
    double f0 = 0.0, f1 = 0.0;
    for (int t = 0; t < pr->shape[2]; ++t)
        for (int k = 0; k < pr->shape[3]; ++k) {
            const double v = c[L.off[3] + k];
            f0 = fmax(f0, fabs(v * L.cth[t]));
            f1 = fmax(f1, fabs(v * L.sth[t]));
        }
    alpha[0] = f0;
    alpha[1] = f1;
    alpha[2] = AT_W;
    alpha[3] = fmax(fabs(AT_AMIN), fabs(AT_AMAX));
    *dt = cfl_step(L, alpha, pr->cfl);
}

int64_t aux_doubles(const Lattice& L) { return (int64_t)(L.coords.size() + L.cth.size() + L.sth.size()); }

// the coordinate vectors, then cos and sin of the theta nodes, to aux (aux_doubles doubles). Pageable sources:
// cudaMemcpyAsync stages them before it returns, so the lattice may go out of scope.
cudaError_t upload_lattice(const Lattice& L, double* aux, cudaStream_t st) {
    cudaError_t e = cudaMemcpyAsync(aux, L.coords.data(), L.coords.size() * sizeof(double), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && !L.cth.empty()) {
        e = cudaMemcpyAsync(aux + L.coords.size(), L.cth.data(), L.cth.size() * sizeof(double), cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(aux + L.coords.size() + L.cth.size(), L.sth.data(), L.sth.size() * sizeof(double),
                                cudaMemcpyHostToDevice, st);
    }
    return e;
}

int check_game(int32_t game, const std::string& fn) {
    if (game != COOPERATIVE && game != ADVERSARIAL && game != CONSTANT)
        return fail(2, fn + ": game must be 0 (cooperative), 1 (adversarial) or 2 (constant)");
    return 0;
}

int game_dissipation(const char* fn, const lsm_hj_problem* problem, int32_t game, double alpha[5], double* dt) {
    Lattice L;
    if (const int rc = check_problem(problem, fn, L)) return rc;
    if (const int rc = check_game(game, fn)) return rc;
    if (!alpha || !dt) return fail(2, std::string(fn) + ": alpha and dt must be non-NULL");
    dissipation(problem, game, L, alpha, dt);
    return 0;
}

int solve(const char* fn_, const lsm_hj_problem* problem, int32_t game, const double* initial, const double* horizons,
          int32_t K, double* out, void* work, void* stream) {
    const std::string fn(fn_);
    Lattice L;
    if (const int rc = check_problem(problem, fn_, L)) return rc;
    if (const int rc = check_game(game, fn)) return rc;
    if (!initial || !horizons || !out || !work)
        return fail(2, fn + ": initial, horizons, out and work must be non-NULL");
    if (K < 1) return fail(2, fn + ": K must be >= 1");
    if ((reinterpret_cast<uintptr_t>(work) % alignof(double)) != 0)
        return fail(2, fn + ": work must be 8-byte aligned");
    for (int32_t k = 0; k < K; ++k) {
        if (!(std::isfinite(horizons[k]) && horizons[k] >= 0.0))
            return fail(2, fn + ": horizons must be finite and >= 0");
        if (k > 0 && horizons[k] < horizons[k - 1]) return fail(2, fn + ": horizons must be non-decreasing");
    }
    double alpha[5], dt;
    dissipation(problem, game, L, alpha, &dt);
    if (!(dt > 0.0 && std::isfinite(dt))) return fail(2, fn + ": the CFL time step is not positive and finite");

    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int64_t cells = L.cells, bytes = cells * (int64_t)sizeof(double);
    double* u0 = static_cast<double*>(work);
    double* u1 = u0 + cells;
    double* u2 = u1 + cells;
    double* aux = u2 + cells;
    cudaError_t e = upload_lattice(L, aux, st);
    if (e != cudaSuccess) return cuda_fail(e, fn + ": upload of the lattice");
    e = cudaMemcpyAsync(u0, initial, bytes, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) return cuda_fail(e, fn + ": copy of the initial values");

    StageParams p{};
    p.coords = aux;
    p.cth = aux + L.coords.size();
    p.sth = p.cth + (problem->dynamics == 1 ? problem->shape[2] : 0);
    p.cells = cells;
    int64_t stride = 1;
    for (int d = L.nd - 1; d >= 0; --d) {
        p.n[d] = problem->shape[d];
        p.stride[d] = stride;
        stride *= problem->shape[d];
        p.coord_off[d] = L.off[d];
        p.inv_dx[d] = 1.0 / L.sp[d];
        p.alpha[d] = alpha[d];
    }
    double tau = 0.0;
    for (int32_t k = 0; k < K; ++k) {
        const double target = horizons[k];
        while (tau < target) {
            double h;
            if (target - tau <= dt) { h = target - tau; tau = target; }
            else { h = dt; tau = tau + dt; }
            const int dyn = problem->dynamics;
            e = game == COOPERATIVE ? launch_game_step<COOPERATIVE>(dyn, p, u0, u1, u2, h, st)
              : game == ADVERSARIAL ? launch_game_step<ADVERSARIAL>(dyn, p, u0, u1, u2, h, st)
                                    : launch_game_step<CONSTANT>(dyn, p, u0, u1, u2, h, st);
            if (e != cudaSuccess) return cuda_fail(e, "lsm_hj_stage_kernel");
        }
        e = cudaMemcpyAsync(out + (int64_t)k * cells, u0, bytes, cudaMemcpyDeviceToDevice, st);
        if (e != cudaSuccess) return cuda_fail(e, fn + ": snapshot");
    }
    return 0;
}

}  // namespace

extern "C" {

int lsm_hj_abi_version(void) { return LSM_HJ_ABI_VERSION; }
const char* lsm_hj_last_error(void) { return g_err.c_str(); }

int64_t lsm_hj_work_bytes(const lsm_hj_problem* problem) {
    Lattice L;
    if (check_problem(problem, "lsm_hj_work_bytes", L) != 0) return 0;
    return (3 * L.cells + aux_doubles(L)) * (int64_t)sizeof(double);
}

int lsm_hj_dissipation(const lsm_hj_problem* problem, double alpha[5], double* dt) {
    return game_dissipation("lsm_hj_dissipation", problem, COOPERATIVE, alpha, dt);
}

int lsm_hj_game_dissipation(const lsm_hj_problem* problem, int32_t game, double alpha[5], double* dt) {
    return game_dissipation("lsm_hj_game_dissipation", problem, game, alpha, dt);
}

int lsm_hj_solve(const lsm_hj_problem* problem, const double* initial, const double* horizons, int32_t K, double* out,
                 void* work, void* stream) {
    return solve("lsm_hj_solve", problem, COOPERATIVE, initial, horizons, K, out, work, stream);
}

int lsm_hj_game_solve(const lsm_hj_problem* problem, int32_t game, const double* initial, const double* horizons,
                      int32_t K, double* out, void* work, void* stream) {
    return solve("lsm_hj_game_solve", problem, game, initial, horizons, K, out, work, stream);
}

int64_t lsm_hj_ttr_work_bytes(const lsm_hj_ttr_problem* problem) {
    Lattice L;
    if (check_ttr_problem(problem, "lsm_hj_ttr_work_bytes", L) != 0) return 0;
    return (3 * L.cells + aux_doubles(L)) * (int64_t)sizeof(double);
}

int lsm_hj_ttr_dissipation(const lsm_hj_ttr_problem* problem, double alpha[4], double* dt) {
    Lattice L;
    if (const int rc = check_ttr_problem(problem, "lsm_hj_ttr_dissipation", L)) return rc;
    if (!alpha || !dt) return fail(2, "lsm_hj_ttr_dissipation: alpha and dt must be non-NULL");
    ttr_dissipation(problem, L, alpha, dt);
    return 0;
}

int lsm_hj_ttr_solve(const lsm_hj_ttr_problem* problem, const double* target, double horizon, double* ttr,
                     double* final_values, void* work, void* stream) {
    Lattice L;
    if (const int rc = check_ttr_problem(problem, "lsm_hj_ttr_solve", L)) return rc;
    if (!target || !ttr || !work) return fail(2, "lsm_hj_ttr_solve: target, ttr and work must be non-NULL");
    if ((reinterpret_cast<uintptr_t>(work) % alignof(double)) != 0)
        return fail(2, "lsm_hj_ttr_solve: work must be 8-byte aligned");
    if (!(std::isfinite(horizon) && horizon >= 0.0)) return fail(2, "lsm_hj_ttr_solve: horizon must be finite and >= 0");
    double alpha[4], dt;
    ttr_dissipation(problem, L, alpha, &dt);
    if (!(dt > 0.0 && std::isfinite(dt)))
        return fail(2, "lsm_hj_ttr_solve: the CFL time step is not positive and finite");

    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int64_t cells = L.cells, bytes = cells * (int64_t)sizeof(double);
    double* u0 = static_cast<double*>(work);
    double* u1 = u0 + cells;
    double* u2 = u1 + cells;
    double* aux = u2 + cells;
    cudaError_t e = upload_lattice(L, aux, st);
    if (e != cudaSuccess) return cuda_fail(e, "lsm_hj_ttr_solve: upload of the lattice");
    e = cudaMemcpyAsync(u0, target, bytes, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) return cuda_fail(e, "lsm_hj_ttr_solve: copy of the target");
    const unsigned grid = (unsigned)((cells + BLOCK - 1) / BLOCK);
    lsm_hj_ttr_init_kernel<<<grid, BLOCK, 0, st>>>(u0, ttr, cells);     // from the copy: ttr may alias target
    if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e, "lsm_hj_ttr_init_kernel");

    TtrParams p{};
    p.ttr = ttr;
    p.coords = aux;
    p.cth = aux + L.coords.size();
    p.sth = p.cth + problem->shape[2];
    p.cells = cells;
    int64_t stride = 1;
    for (int d = 3; d >= 0; --d) {
        p.n[d] = problem->shape[d];
        p.stride[d] = stride;
        stride *= problem->shape[d];
        p.coord_off[d] = L.off[d];
        p.inv_dx[d] = 1.0 / L.sp[d];
        p.alpha[d] = alpha[d];
    }
    double tau = 0.0;
    while (tau < horizon) {
        const double tau0 = tau;
        double h;
        if (horizon - tau <= dt) { h = horizon - tau; tau = horizon; }
        else { h = dt; tau = tau + dt; }
        if ((e = launch_ttr_step(p, u0, u1, u2, tau0, h, st)) != cudaSuccess) return cuda_fail(e, "lsm_hj_ttr_stage_kernel");
    }
    if (final_values) {
        e = cudaMemcpyAsync(final_values, u0, bytes, cudaMemcpyDeviceToDevice, st);
        if (e != cudaSuccess) return cuda_fail(e, "lsm_hj_ttr_solve: copy of the final values");
    }
    return 0;
}

}  // extern "C"

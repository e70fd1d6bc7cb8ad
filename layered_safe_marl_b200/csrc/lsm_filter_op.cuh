// lsm_filter_op.cuh - the HJ safety filter as a standalone batched operator (lsm_safety_filter / lsm_hj_lookup).
//
// The same device code the specialised step pipeline runs, applied to states the caller owns instead of the env's:
//   relative state   relative_state_rot (one sincos per ego; identical to the literal form for the double integrator)
//   HJ value         pair_value_rel: corner-packed table when the handle built one, else the scattered stencil
//   filter           filter_resolve (gradient, least-restrictive bang-bang below 0.4 or CBF-QP, clipping, filtered flag)
//   gradient         grid_grad: float4 rows (4-D) / padded rows (5-D, built for every handle by lsm_set_value_grid)
// F32 = LSM_FLAG_INTERP_FLOAT32 of the handle, chosen at compile time like the agent and pair kernels.
//
// lsm_safety_filter_kernel: a block owns kFopRows rows at a time. Phase 1: kFopLanes threads per row evaluate distance and
// HJ value of kFopLanes slots at once (a thread per (row, slot), as lsm_pair_kernel does), write them to shared memory,
// and the row's owner thread folds them into its running first minimum in ascending slot order (np.argmin); repeated
// over chunks of kFopLanes slots. Phase 2: the owner thread resolves its row (filter_resolve) and writes the outputs.
#pragma once
#include "lsm_kernel_spec.cuh"
#include "lsm_host.h"

namespace lsm {

constexpr int kFopRows = 32;                    // rows per block tile = owner threads (warp 0)
constexpr int kFopLanes = 8;                    // slot lanes per row in phase 1
constexpr int kFopThreads = kFopRows * kFopLanes;
constexpr int kLookupThreads = 128;

template <int DYN, bool F32>
__global__ void __launch_bounds__(kFopThreads) lsm_safety_filter_kernel(const __grid_constant__ KParams kp,
                                                                      const __grid_constant__ FilterOpArgs a) {
    constexpr int ND = DYN == LSM_DYN_DOUBLE_INTEGRATOR ? 4 : 5;
    // [lane][row]: the owner thread of row r reads s_*[k][r], conflict-free across the owner warp
    __shared__ double s_v[kFopLanes][kFopRows];
    __shared__ double s_d2[kFopLanes][kFopRows];
    __shared__ unsigned char s_on[kFopLanes][kFopRows];
    const int tid = threadIdx.x;
    const int tr = tid / kFopLanes, tk = tid - tr * kFopLanes;     // phase 1: row and slot lane of this thread
    const long long tiles = (a.rows + kFopRows - 1) / kFopRows;
    const int M = a.slots;
    for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const long long row0 = tile * kFopRows;
        // phase-1 row of this thread
        const long long prow = row0 + tr;
        const bool prow_on = prow < a.rows;
        double ex = 0.0, ey = 0.0, e2 = 0.0, e3 = 0.0, se = 0.0, ce = 1.0, psep = kp.vg.separation_distance;
        if (prow_on) {
            const double* e = a.ego + (size_t)prow * 4;
            ex = e[0]; ey = e[1]; e2 = e[2]; e3 = e[3];
            if constexpr (DYN != LSM_DYN_DOUBLE_INTEGRATOR) lsm_sincos(e2, &se, &ce);
            if (a.sep != nullptr) psep = a.sep[prow];
        }
        // owner state (tid < kFopRows): first minimum of distance and value over the active slots so far
        int kv = -1;
        double best_d2 = 0.0, best_v = 0.0;
        for (int c = 0; c < M; c += kFopLanes) {
            const int slot = c + tk;
            bool on = false;
            double v = INFINITY, d2 = 0.0;
            if (prow_on && slot < M) {
                const size_t s = (size_t)prow * M + slot;
                on = a.active == nullptr || a.active[s] != 0;
                if (on) {
                    const double* o = a.others + s * 4;
                    const double ox = o[0], oy = o[1], o2 = o[2], o3 = o[3];
                    const double ddx = ox - ex, ddy = oy - ey;
                    d2 = ddx * ddx + ddy * ddy;
                    double rel[ND];
                    relative_state_rot_sc<DYN>(ex, ey, e2, e3, ox, oy, o2, o3, se, ce, rel);
                    v = shift_value(pair_value_rel<ND, kPeriodicRuntime, F32>(kp.vg, rel), psep, kp.vg);
                }
            }
            s_v[tk][tr] = v; s_d2[tk][tr] = d2; s_on[tk][tr] = on ? 1 : 0;
            __syncthreads();
            if (tid < kFopRows) {
                // np.argmin semantics: ascending slot order, strict comparison keeps the first minimum (a NaN distance
                // that comes first stays, as in the sequential scan of the reference)
#pragma unroll
                for (int k = 0; k < kFopLanes; ++k) {
                    if (!s_on[k][tid]) continue;
                    const double dk = s_d2[k][tid], vk = s_v[k][tid];
                    const bool first = kv < 0;
                    if (first || dk < best_d2) best_d2 = dk;      // only the smallest distance is used (range test)
                    if (first || vk < best_v) { kv = c + k; best_v = vk; }
                }
            }
            __syncthreads();
        }
        // phase 2: the owner thread resolves its row
        const long long row = row0 + tid;
        if (tid < kFopRows && row < a.rows) {
            const double* e = a.ego + (size_t)row * 4;
            const double rx = e[0], ry = e[1], r2 = e[2], r3 = e[3];
            const double raw0 = a.ego_action[(size_t)row * 2], raw1 = a.ego_action[(size_t)row * 2 + 1];
            double safe0 = raw0, safe1 = raw1;
            int filt = 0;
            if (kv >= 0) {
                const double* o = a.others + ((size_t)row * M + kv) * 4;
                const double* ou = a.other_actions + ((size_t)row * M + kv) * 2;
                double rse = 0.0, rce = 1.0;
                if constexpr (DYN != LSM_DYN_DOUBLE_INTEGRATOR) lsm_sincos(r2, &rse, &rce);
                filter_resolve<DYN, true, F32>(kp, sqrt(best_d2), best_v, !isinf(best_v), rx, ry, r2, r3, o[0], o[1], o[2], o[3],
                                               raw0, raw1, ou[0], ou[1], safe0, safe1, filt, rse, rce);
            }
            a.safe_action[(size_t)row * 2] = safe0;
            a.safe_action[(size_t)row * 2 + 1] = safe1;
            if (a.filtered != nullptr) a.filtered[row] = (uint8_t)filt;
            if (a.index != nullptr) a.index[row] = kv;
            if (a.value != nullptr) a.value[row] = kv >= 0 ? best_v : INFINITY;
        }
    }
}

// get_value_of_relative_state (safety_filter.py:192-201, 345-354) and the gradient (safety_filter.py:245, 418): one
// thread per point
template <int DYN, bool F32>
__global__ void __launch_bounds__(kLookupThreads) lsm_hj_lookup_kernel(const __grid_constant__ KParams kp,
                                                                     const __grid_constant__ LookupArgs a) {
    constexpr int ND = DYN == LSM_DYN_DOUBLE_INTEGRATOR ? 4 : 5;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < a.points; k += stride) {
        double rel[ND];
        if (a.rel != nullptr) {
#pragma unroll
            for (int d = 0; d < ND; ++d) rel[d] = a.rel[(size_t)k * ND + d];
        } else {
            const double* e = a.ego + (size_t)k * 4;
            const double* o = a.other + (size_t)k * 4;
            relative_state_rot<DYN>(e[0], e[1], e[2], e[3], o[0], o[1], o[2], o[3], rel);
        }
        const double sep = a.sep != nullptr ? a.sep[k] : kp.vg.separation_distance;
        a.value[k] = shift_value(pair_value_rel<ND, kPeriodicRuntime, F32>(kp.vg, rel), sep, kp.vg);
        if (a.grad != nullptr) {
            // a NaN coordinate makes every component NaN (Grid.interpolate); any other point, inside the box or not, is
            // interpolated with the declared index clamp / wrap
            bool nan_pos = false;
#pragma unroll
            for (int d = 0; d < ND; ++d) nan_pos = nan_pos || isnan(rel[d]);
            double g[ND];
            if (nan_pos) {
#pragma unroll
                for (int d = 0; d < ND; ++d) g[d] = NAN;
            } else grid_grad<ND, F32>(kp.vg, rel, g);
#pragma unroll
            for (int d = 0; d < ND; ++d) a.grad[(size_t)k * ND + d] = g[d];
        }
        if (a.rel_out != nullptr) {
#pragma unroll
            for (int d = 0; d < ND; ++d) a.rel_out[(size_t)k * ND + d] = rel[d];
        }
    }
}

}  // namespace lsm

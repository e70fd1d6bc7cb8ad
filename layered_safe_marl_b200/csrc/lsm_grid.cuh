// lsm_grid.cuh - the HJ grid lookups of every kernel: multilinear interpolation on a regular grid (hj_reachability
// Grid.interpolate, declared semantics: DESIGN.md "grid interpolation"), in float64 and in float32 (LSM_FLAG_INTERP_FLOAT32),
// and the builders of the library-owned grid copies (corner-packed values, padded 5-D gradient rows).
//
// The contract, stated once for both arithmetics (the oracle's interpolate / interpolate_f32):
//   * position pos = (x - lo) / spacing per dimension (GridArith: the only place the two arithmetics differ, together with
//     the clamp); a NaN position makes the lookup invalid;
//   * the declared clamp of pos to [-1e9, 1e9], floor, weights (1 - w, w);
//   * indices: lower = floor(pos), upper = lower + 1, both wrapped on periodic dimensions, clamped to [0, n - 1] on the
//     others; 32-bit cell indices (fill_grid refuses grids of 2^31 cells or more);
//   * corners in binary counting order, dimension 0 slowest; weight ((w0 * w1) * w2) ..; sequential corner sum, no FMA
//     (-fmad=false). Weights, products and sums are float64, or float32 in the float32 arithmetic.
#pragma once
#include "lsm_device.cuh"

namespace lsm {

// exactly rounded a / b through the precomputed reciprocal y = RN(1/b) (Markstein: q0 = a*y, r = fma(-b,q0,a),
// q = fma(r,y,q0) equals RN(a/b); checked on the CPU in tests/test_host_logic.py)
__device__ __forceinline__ double div_exact(double a, double b, double y /* RN(1/b) */) {
    const double q0 = a * y;
    const double r = fma(-b, q0, a);
    return fma(r, y, q0);
}

// periodic grid index: i mod n in [0, n). In-grid states land in [0, n) (an angle difference wrapped to one period), so the
// integer division (~30 instructions) sits behind an "already in range" test. Measured on B200 (same-box A/B,
// profiles/experiments/r02_wrap_index_ab.txt): for the 5-D airtaxi grid one shared out-of-line copy is faster (cfg3 352.7
// -> 348.7 us; the unrolled 32-corner stencils are bound by instruction fetch), for the 4-D grids the call costs the
// pair kernel six registers and a stack frame (cfg2 back-to-back 40.4 -> 43.2 us), so those keep it inline.
__device__ __noinline__ int wrap_index_slow(int i, int n) { i %= n; if (i < 0) i += n; return i; }
template <bool OUT_OF_LINE>
__device__ __forceinline__ int wrap_index(int i, int n) {
    if constexpr (OUT_OF_LINE) return ((unsigned)i < (unsigned)n) ? i : wrap_index_slow(i, n);
    else { if ((unsigned)i >= (unsigned)n) { i %= n; if (i < 0) i += n; } return i; }
}

// The two arithmetics: grid position and declared clamp.
//   float64: exactly rounded division through the reciprocal (div_exact);
//   float32: state, lo and spacing rounded to float32, IEEE float32 division (what jax computes without x64).
template <bool F32>
struct GridArith {
    using W = double;
    __device__ __forceinline__ static double pos(const GridDev& g, double x, int d) {
        return div_exact(x - g.lo[d], g.spacing[d], g.inv_spacing[d]);
    }
    __device__ __forceinline__ static double clamp(double p) { return !(fabs(p) <= 1.0e9) ? (p < 0.0 ? -1.0e9 : 1.0e9) : p; }
};
template <>
struct GridArith<true> {
    using W = float;
    __device__ __forceinline__ static float pos(const GridDev& g, double x, int d) {
        return __fdiv_rn((float)x - (float)g.lo[d], (float)g.spacing[d]);
    }
    __device__ __forceinline__ static float clamp(float p) { return fminf(fmaxf(p, -1.0e9f), 1.0e9f); }
};

// dimension d of x: the weights of the lower / upper node and the lower node index before wrap or clamp; `valid` drops
// to false for a NaN position
template <bool F32>
__device__ __forceinline__ int grid_axis(const GridDev& g, double x, int d, typename GridArith<F32>::W& wlo,
                                         typename GridArith<F32>::W& whi, bool& valid) {
    using A = GridArith<F32>;
    typename A::W pos = A::pos(g, x, d);
    if (isnan(pos)) valid = false;
    pos = A::clamp(pos);                          // never taken in-grid
    const typename A::W fl = floor(pos);
    whi = pos - fl;
    wlo = (typename A::W)1 - whi;
    return (int)fl;                               // |fl| <= 1e9 fits in int32
}

// weight of one corner: ((w0 * w1) * w2) .., dimension 0 first
template <int ND, class W>
__device__ __forceinline__ W corner_weight(const W (&wlo)[ND], const W (&whi)[ND], int corner) {
    W weight = 0;
#pragma unroll
    for (int d = 0; d < ND; ++d) {
        const W wd = ((corner >> (ND - 1 - d)) & 1) ? whi[d] : wlo[d];
        weight = (d == 0) ? wd : weight * wd;
    }
    return weight;
}

template <int ND, bool F32>
struct GridStencil {
    using W = typename GridArith<F32>::W;
    int lo[ND], hi[ND];        // linear offset contributions of the lower / upper node per dimension
    W wlo[ND], whi[ND];
    bool valid;
};

template <int ND, bool F32>
__device__ __forceinline__ void grid_setup(const GridDev& g, const double (&x)[ND], GridStencil<ND, F32>& s) {
    s.valid = true;
    int mul = 1;
#pragma unroll
    for (int d = ND - 1; d >= 0; --d) {
        int il = grid_axis<F32>(g, x[d], d, s.wlo[d], s.whi[d], s.valid), ih = il + 1;
        const int n = g.shape[d];
        if (g.periodic[d]) {
            il = wrap_index<(ND == 5)>(il, n);
            ih = il + 1 == n ? 0 : il + 1;          // (il + 1) mod n
        } else {
            il = min(max(il, 0), n - 1);
            ih = min(max(ih, 0), n - 1);
        }
        s.lo[d] = il * mul; s.hi[d] = ih * mul;
        mul *= n;
    }
}

// value: all 2^ND loads are issued first (one memory round trip per lookup instead of 2^ND dependent ones), then the
// sequential corner sum
template <int ND, bool F32>
__device__ __forceinline__ double corner_value_sum(const GridDev& g, const GridStencil<ND, F32>& s) {
    using W = typename GridArith<F32>::W;
    constexpr int NC = 1 << ND;
    float v[NC];
    const unsigned long long keep = l2_evict_last();
#pragma unroll
    for (int corner = 0; corner < NC; ++corner) {
        int lin = 0;
#pragma unroll
        for (int d = 0; d < ND; ++d) lin += ((corner >> (ND - 1 - d)) & 1) ? s.hi[d] : s.lo[d];
        v[corner] = ldg_hint(g.values + lin, keep);
    }
    W acc = 0;
#pragma unroll
    for (int corner = 0; corner < NC; ++corner) acc = acc + corner_weight<ND>(s.wlo, s.whi, corner) * (W)v[corner];
    return (double)acc;
}

// all gradient components in one pass over the corners (same corner / weight order as the value): one float4 row per
// corner for 4-D grids, the padded rows (GridDev::grads8, two float4) for 5-D grids. The float32 arithmetic gives NaN
// components for a NaN position, as the oracle's interpolate_f32 does.
template <int ND, bool F32>
__device__ __forceinline__ void corner_grad_sum(const GridDev& g, const GridStencil<ND, F32>& s, double (&out)[ND]) {
    static_assert(ND == 4 || ND == 5, "the HJ value grids are 4-D or 5-D");
    using W = typename GridArith<F32>::W;
    W acc[ND];
#pragma unroll
    for (int d = 0; d < ND; ++d) acc[d] = 0;
    const unsigned long long keep = l2_evict_last();
#pragma unroll
    for (int corner = 0; corner < (1 << ND); ++corner) {
        const W weight = corner_weight<ND>(s.wlo, s.whi, corner);
        int lin = 0;
#pragma unroll
        for (int d = 0; d < ND; ++d) lin += ((corner >> (ND - 1 - d)) & 1) ? s.hi[d] : s.lo[d];
        if constexpr (ND == 4) {
            const float4 v = ldg_hint(reinterpret_cast<const float4*>(g.grads) + lin, keep);
            acc[0] = acc[0] + weight * (W)v.x; acc[1] = acc[1] + weight * (W)v.y;
            acc[2] = acc[2] + weight * (W)v.z; acc[3] = acc[3] + weight * (W)v.w;
        } else {
            const float4 a = ldg_hint(reinterpret_cast<const float4*>(g.grads8) + 2 * (size_t)lin, keep);
            const float4 b = ldg_hint(reinterpret_cast<const float4*>(g.grads8) + 2 * (size_t)lin + 1, keep);
            acc[0] = acc[0] + weight * (W)a.x; acc[1] = acc[1] + weight * (W)a.y;
            acc[2] = acc[2] + weight * (W)a.z; acc[3] = acc[3] + weight * (W)a.w;
            acc[ND - 1] = acc[ND - 1] + weight * (W)b.x;
        }
    }
#pragma unroll
    for (int d = 0; d < ND; ++d) out[d] = (F32 && !s.valid) ? (double)NAN : (double)acc[d];
}

// interpolated value at x; NaN for a NaN position
template <int ND, bool F32>
__device__ __forceinline__ double grid_value(const GridDev& g, const double (&x)[ND]) {
    GridStencil<ND, F32> s;
    grid_setup<ND, F32>(g, x, s);
    return s.valid ? corner_value_sum<ND, F32>(g, s) : NAN;
}

// interpolated gradient at x
template <int ND, bool F32>
__device__ __forceinline__ void grid_grad(const GridDev& g, const double (&x)[ND], double (&out)[ND]) {
    GridStencil<ND, F32> s;
    grid_setup<ND, F32>(g, x, s);
    corner_grad_sum<ND, F32>(g, s, out);
}

// grid_value out of line. The point arrives as scalars (x4 unused for ND == 4): an array reference would put the
// caller's array in local memory.
template <int ND, bool F32>
__device__ __noinline__ double grid_value_noinline(const GridDev& g, double x0, double x1, double x2, double x3, double x4) {
    double x[ND];
    x[0] = x0; x[1] = x1; x[2] = x2; x[3] = x3;
    if constexpr (ND == 5) x[4] = x4;
    return grid_value<ND, F32>(g, x);
}

// grid_grad out of line, the components returned by value
template <int ND>
struct GridGrad { double d[ND]; };
template <int ND, bool F32>
__device__ __noinline__ GridGrad<ND> grid_grad_noinline(const GridDev& g, double x0, double x1, double x2, double x3, double x4) {
    double x[ND];
    x[0] = x0; x[1] = x1; x[2] = x2; x[3] = x3;
    if constexpr (ND == 5) x[4] = x4;
    GridGrad<ND> r;
    grid_grad<ND, F32>(g, x, r.d);
    return r;
}

// The generic kernel's lookups: the handle's arithmetic (GridDev::f32) chosen at run time between the two out-of-line
// instantiations, so that the fused kernel (~250 registers) inlines neither.
template <int ND>
__device__ __forceinline__ double grid_value_rt(const GridDev& g, const double (&x)[ND]) {
    const double x4 = ND == 5 ? x[ND - 1] : 0.0;
    return g.f32 ? grid_value_noinline<ND, true>(g, x[0], x[1], x[2], x[3], x4)
                 : grid_value_noinline<ND, false>(g, x[0], x[1], x[2], x[3], x4);
}
template <int ND>
__device__ __forceinline__ void grid_grad_rt(const GridDev& g, const double (&x)[ND], double (&out)[ND]) {
    const double x4 = ND == 5 ? x[ND - 1] : 0.0;
    const GridGrad<ND> r = g.f32 ? grid_grad_noinline<ND, true>(g, x[0], x[1], x[2], x[3], x4)
                                 : grid_grad_noinline<ND, false>(g, x[0], x[1], x[2], x[3], x4);
#pragma unroll
    for (int d = 0; d < ND; ++d) out[d] = r.d[d];
}

// padded 5-D gradient rows (GridDev::grads8): 5 floats -> 8, so that one corner is two 16-byte loads
__global__ void __launch_bounds__(256) lsm_pad_grads_kernel(const float* __restrict__ grads, float* __restrict__ grads8, long long cells) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= cells * 8) return;
    const long long cell = t >> 3; const int d = (int)(t & 7);
    grads8[t] = d < 5 ? grads[cell * 5 + d] : 0.0f;
}

// ---------------------------------------------------------------------------------------------
// corner-packed table (GridDev::packed): builder + lookup. The lookup reproduces grid_value bit for bit (same positions,
// weights, corner order, sequential adds), including the declared index clamp outside the box; only NaN positions take
// the scattered path.
// ---------------------------------------------------------------------------------------------
// Table extent per dim: n on periodic dims; n + 1 on the others, slot c standing for the index pair
// (max(c - 1, 0), min(c, n - 1)) - slot 0 is the "both clamped to node 0" pair the declared out-of-box behaviour needs,
// slot n the "both clamped to node n - 1" pair - so every finite position is served by one chunk.
template <int ND>
__global__ void __launch_bounds__(256) lsm_pack_grid_kernel(const float* __restrict__ values, float* __restrict__ packed,
                                                          GridDev g, long long cells) {
    constexpr int NC = 1 << ND;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= cells * NC) return;
    const long long cell = t / NC; const int corner = (int)(t - cell * NC);
    long long rem = cell, lin = 0, mul = 1;
#pragma unroll
    for (int d = ND - 1; d >= 0; --d) {
        const int n = g.shape[d];
        const int ext = g.periodic[d] ? n : n + 1;
        const int c = (int)(rem % ext); rem /= ext;
        int il, ih;
        if (g.periodic[d]) { il = c; ih = c + 1 >= n ? c + 1 - n : c + 1; }
        else { il = c - 1 < 0 ? 0 : c - 1; ih = c > n - 1 ? n - 1 : c; }
        lin += (long long)(((corner >> (ND - 1 - d)) & 1) ? ih : il) * mul;
        mul *= n;
    }
    packed[t] = values[lin];
}

// Which dimensions of a lookup wrap. kPeriodicRuntime reads GridDev::periodic (any grid); any other value is a
// compile-time mask (bit d = dimension d is periodic), so the per-dimension branch and the inline integer modulo of the
// dimensions that cannot wrap are not in the code at all. The pair kernel is instantiated for the mask of the grids the
// specialised shapes are built for (kPairPeriodic) and falls back to the run-time form for any other grid.
constexpr int kPeriodicRuntime = -1;
template <int PER>
__device__ __forceinline__ bool dim_periodic(const GridDev& g, int d) {
    if constexpr (PER == kPeriodicRuntime) return g.periodic[d] != 0;
    else return ((PER >> d) & 1) != 0;
}
// double integrator: no periodic dimension; airtaxi: the relative heading, dimension 2 (hj_grid.py)
template <int DYN>
constexpr int kPairPeriodic = DYN == LSM_DYN_DOUBLE_INTEGRATOR ? 0 : 1 << 2;

// grid_value from the corner-packed table; false only for NaN positions. The slot c = clamp(floor, -1, n - 1) + 1 stands
// for the clamped index pair (non-periodic dims), the wrapped lower index il for the pair (il, (il + 1) mod n).
template <int ND, int PER, bool F32>
__device__ __forceinline__ bool packed_value(const GridDev& g, const double (&x)[ND], double& out) {
    using W = typename GridArith<F32>::W;
    constexpr int NC = 1 << ND;
    W wlo[ND], whi[ND];
    bool ok = true;
    int cell = 0, mul = 1;
#pragma unroll
    for (int d = ND - 1; d >= 0; --d) {
        const int fl = grid_axis<F32>(g, x[d], d, wlo[d], whi[d], ok);
        const int n = g.shape[d];
        if (dim_periodic<PER>(g, d)) {
            cell += wrap_index<(ND == 5)>(fl, n) * mul; mul *= n;
        } else {
            cell += (min(max(fl, -1), n - 1) + 1) * mul; mul *= n + 1;
        }
    }
    if (!ok) return false;
    const float4* src = reinterpret_cast<const float4*>(g.packed) + (size_t)cell * (NC / 4);
    float v[NC];
#pragma unroll
    for (int k = 0; k < NC / 4; ++k) {
        const float4 q = __ldg(src + k);
        v[4 * k] = q.x; v[4 * k + 1] = q.y; v[4 * k + 2] = q.z; v[4 * k + 3] = q.w;
    }
    W acc = 0;
#pragma unroll
    for (int corner = 0; corner < NC; ++corner) acc = acc + corner_weight<ND>(wlo, whi, corner) * (W)v[corner];
    out = (double)acc;
    return true;
}

// raw (unshifted) HJ value of a relative state for the specialised pipeline and the operator: the corner-packed table
// when the handle built one, else the scattered stencil; +inf = outside the declared range / NaN
template <int ND, int PER, bool F32>
__device__ __forceinline__ double pair_value_rel(const GridDev& vg, const double (&rel)[ND]) {
    if (vg.packed != nullptr) {
        double v;
        if (packed_value<ND, PER, F32>(vg, rel, v)) return isnan(v) ? INFINITY : v;
    }
    const double v = grid_value_noinline<ND, F32>(vg, rel[0], rel[1], rel[2], rel[3], ND == 5 ? rel[ND - 1] : 0.0);
    return isnan(v) ? INFINITY : v;
}

}  // namespace lsm

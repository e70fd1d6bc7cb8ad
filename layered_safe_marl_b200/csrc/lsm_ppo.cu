// lsm_ppo.cu - the PPO-input kernels declared in include/lsm_b200_ppo.h (liblsm_b200_ppo.so).
//
// lsm_returns_kernel: one thread per column walks t = T-1 .. 0 and replays DeviceGraphRolloutBuffer.compute_returns'
// torch loop with every operation rounded once (__fmul_rn / __fadd_rn / __fsub_rn; the library is built with
// -fmad=false as well). The loads of a step do not depend on the recursion, so they are issued a chunk of P steps ahead
// into a second register set while the current chunk is computed: with few warps per SM (C = 32 768 columns are 1 024
// warps, about 7 per SM of a B200) the latency has to be hidden by loads in flight rather than by occupancy.
//
// The advantage moments are accumulated per thread in float64 as sums shifted by the thread's first active value (no
// cancellation when the mean is far from zero), turned into (count, mean, M2), merged with Chan's formula in a fixed
// shuffle order, written per block to scratch, and merged in a fixed order by a one-block kernel. No atomics, so two
// calls on one device give the same bits.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>
#include <string>
#include <utility>

#include "../../include/lsm_b200_ppo.h"

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) { g_err = msg; return code; }
int cuda_fail(cudaError_t e, const char* what) {
    g_err = std::string(what) + ": " + cudaGetErrorString(e);
    return 100 + (int)e;
}

constexpr int P = 8;                    // steps per chunk: loads run 8-16 steps ahead of the recursion
constexpr int FINAL_THREADS = 1024;     // threads of the one-block final merge
constexpr int MAX_BLOCK = 128;

struct ReturnsParams {
    int64_t T, C;
    const float* rewards;
    float* value_preds;
    const float* next_value;
    const float* masks;
    const float* bad_masks;
    float* returns;
    float* advantages;
    const float* active_masks;
    const float* value_scale;
    const float* value_shift;
    double* partials;                   // [gridDim.x][3] count, mean, M2
    float gamma, gamma_lambda;
};

struct Chunk { float r[P], v[P], m[P], b[P], a[P]; };

// read-once streams: evict-first loads
__device__ __forceinline__ float ld(const float* p) { return __ldcs(p); }

template <bool GAE, bool PTL, bool NEED_V, bool MOM>
__device__ __forceinline__ void load_chunk(Chunk& ch, const ReturnsParams& p, int64_t t0, int64_t c) {
    const int64_t C = p.C;
#pragma unroll
    for (int k = 0; k < P; ++k) {
        const int64_t t = t0 - k;
        if (t >= 0) {
            const int64_t o = t * C + c;
            ch.r[k] = ld(p.rewards + o);
            ch.m[k] = ld(p.masks + o + C);
            if (NEED_V) ch.v[k] = ld(p.value_preds + o);
            if (PTL) ch.b[k] = ld(p.bad_masks + o + C);
            if (MOM) ch.a[k] = ld(p.active_masks + o);
        }
    }
}

// Chan et al.'s pairwise merge of (count, mean, M2); an empty side leaves the other unchanged
__device__ __forceinline__ void merge(double& n, double& m, double& M, double nb, double mb, double Mb) {
    if (nb == 0.0) return;
    if (n == 0.0) { n = nb; m = mb; M = Mb; return; }
    const double nn = __dadd_rn(n, nb);
    const double d = __dsub_rn(mb, m);
    m = __dadd_rn(m, __dmul_rn(d, __ddiv_rn(nb, nn)));
    M = __dadd_rn(__dadd_rn(M, Mb), __dmul_rn(__dmul_rn(d, d), __ddiv_rn(__dmul_rn(n, nb), nn)));
    n = nn;
}

// fixed-order merge of a block's per-thread moments; thread 0 returns the block's
__device__ __forceinline__ void block_merge(double& n, double& m, double& M) {
    __shared__ double sh[3][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const double nb = __shfl_down_sync(0xffffffffu, n, off);
        const double mb = __shfl_down_sync(0xffffffffu, m, off);
        const double Mb = __shfl_down_sync(0xffffffffu, M, off);
        if (lane + off < 32) merge(n, m, M, nb, mb, Mb);
    }
    const int warps = (blockDim.x + 31) >> 5;
    if (warps == 1) return;
    if (lane == 0) { sh[0][warp] = n; sh[1][warp] = m; sh[2][warp] = M; }
    __syncthreads();
    if (threadIdx.x == 0)
        for (int w = 1; w < warps; ++w) merge(n, m, M, sh[0][w], sh[1][w], sh[2][w]);
}

template <bool GAE, bool PTL, bool DENORM, bool ADV, bool MOM>
__global__ void __launch_bounds__(MAX_BLOCK) lsm_returns_kernel(const ReturnsParams p) {
    constexpr bool NEED_V = GAE || (PTL && !GAE) || ADV || MOM;
    const int64_t C = p.C, T = p.T;
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double cnt = 0.0, shift0 = 0.0, s1 = 0.0, s2 = 0.0;
    if (c < C) {
        const float scale = DENORM ? *p.value_scale : 1.0f, shift = DENORM ? *p.value_shift : 0.0f;
        const float gamma = p.gamma, gl = p.gamma_lambda;
        const float nv = p.next_value[c];
        float carry;                    // GAE: d(value_preds[t+1]); discounted: returns[t+1]
        if (GAE) {
            p.value_preds[T * C + c] = nv;
            carry = DENORM ? __fadd_rn(__fmul_rn(nv, scale), shift) : nv;
        } else {
            p.returns[T * C + c] = nv;
            carry = nv;
        }
        float gae = 0.0f;
        Chunk cur, nxt;
        load_chunk<GAE, PTL, NEED_V, MOM>(cur, p, T - 1, c);
        for (int64_t t0 = T - 1; t0 >= 0; t0 -= P) {
            load_chunk<GAE, PTL, NEED_V, MOM>(nxt, p, t0 - P, c);
#pragma unroll
            for (int k = 0; k < P; ++k) {
                const int64_t t = t0 - k;
                if (t < 0) break;
                const float r = cur.r[k], m = cur.m[k];
                float dv = 0.0f;
                if (NEED_V) dv = DENORM ? __fadd_rn(__fmul_rn(cur.v[k], scale), shift) : cur.v[k];
                float ret;
                if (GAE) {
                    // delta = r + gamma * d(v[t+1]) * m[t+1] - d(v[t]);  gae = delta + gamma_lambda * m[t+1] * gae
                    const float delta = __fsub_rn(__fadd_rn(r, __fmul_rn(__fmul_rn(gamma, carry), m)), dv);
                    gae = __fadd_rn(delta, __fmul_rn(__fmul_rn(gl, m), gae));
                    if (PTL) gae = __fmul_rn(gae, cur.b[k]);
                    ret = __fadd_rn(gae, dv);
                    carry = dv;
                } else {
                    // r = returns[t+1] * gamma * m[t+1] + r;  r = r * b + (1 - b) * d(v[t])
                    ret = __fadd_rn(__fmul_rn(__fmul_rn(carry, gamma), m), r);
                    if (PTL) ret = __fadd_rn(__fmul_rn(ret, cur.b[k]), __fmul_rn(__fsub_rn(1.0f, cur.b[k]), dv));
                    carry = ret;
                }
                const int64_t o = t * C + c;
                p.returns[o] = ret;
                if (ADV || MOM) {
                    const float adv = __fsub_rn(ret, dv);
                    if (ADV) __stcs(p.advantages + o, adv);
                    if (MOM) {
                        const bool act = cur.a[k] != 0.0f;
                        const double x = (double)adv;
                        shift0 = (act && cnt == 0.0) ? x : shift0;
                        const double y = __dsub_rn(x, shift0);
                        cnt = act ? __dadd_rn(cnt, 1.0) : cnt;
                        s1 = act ? __dadd_rn(s1, y) : s1;
                        s2 = act ? __dadd_rn(s2, __dmul_rn(y, y)) : s2;
                    }
                }
            }
            cur = nxt;
        }
    }
    if (MOM) {
        // shifted sums -> (count, mean, M2) of this column
        double n = cnt, m = 0.0, M = 0.0;
        if (n > 0.0) {
            m = __dadd_rn(shift0, __ddiv_rn(s1, n));
            M = fmax(__dsub_rn(s2, __ddiv_rn(__dmul_rn(s1, s1), n)), 0.0);
        }
        block_merge(n, m, M);
        if (threadIdx.x == 0) {
            double* out = p.partials + 3 * (int64_t)blockIdx.x;
            out[0] = n; out[1] = m; out[2] = M;
        }
    }
}

// one block: merge the per-block partials in a fixed order -> stats64 {count, mean, std}, stats {mean, std}
__global__ void __launch_bounds__(FINAL_THREADS) lsm_returns_moments_kernel(const double* partials, int64_t blocks,
                                                                           double* stats64, float* stats) {
    double n = 0.0, m = 0.0, M = 0.0;
    for (int64_t b = threadIdx.x; b < blocks; b += blockDim.x)
        merge(n, m, M, partials[3 * b], partials[3 * b + 1], partials[3 * b + 2]);
    block_merge(n, m, M);
    if (threadIdx.x == 0) {
        double mean = NAN, sd = NAN;
        if (n > 0.0) { mean = m; sd = sqrt(__ddiv_rn(M, n)); }
        if (stats64) { stats64[0] = n; stats64[1] = mean; stats64[2] = sd; }
        if (stats) { stats[0] = __double2float_rn(mean); stats[1] = __double2float_rn(sd); }
    }
}

using Launch = void (*)(const ReturnsParams&, unsigned, unsigned, cudaStream_t);

template <int MODE>
void launch_returns(const ReturnsParams& p, unsigned grid, unsigned block, cudaStream_t s) {
    lsm_returns_kernel<(MODE & 1) != 0, (MODE & 2) != 0, (MODE & 4) != 0, (MODE & 8) != 0, (MODE & 16) != 0>
        <<<grid, block, 0, s>>>(p);
}

template <int... M>
constexpr auto launch_table(std::integer_sequence<int, M...>) {
    struct Table { Launch f[sizeof...(M)]; };
    return Table{{&launch_returns<M>...}};
}
constexpr auto kLaunch = launch_table(std::make_integer_sequence<int, 32>{});

// 32-thread blocks while every column fits in about one wave (spreads C = 32 768 over all 148 SMs: 6-7 warps each),
// 128-thread blocks above (fewer partials to merge, same balance once there are several waves)
int block_threads(int64_t C, int sms) {
    return C <= (int64_t)32 * 8 * sms ? 32 : MAX_BLOCK;
}

int64_t max_blocks(int64_t C) { return (C + 31) / 32; }

int sm_count() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0) return 148;
    if (dev < 64 && cached[dev] > 0) return cached[dev];
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
    if (dev < 64) cached[dev] = sms;
    return sms;
}

}  // namespace

extern "C" {

int lsm_ppo_abi_version(void) { return LSM_PPO_ABI_VERSION; }
const char* lsm_ppo_last_error(void) { return g_err.c_str(); }

int64_t lsm_returns_scratch_bytes(int64_t columns) {
    return 3 * (int64_t)sizeof(double) * (columns > 0 ? max_blocks(columns) : 1);
}

int lsm_compute_returns(const lsm_returns_io* io, void* stream) {
    if (!io) return fail(2, "lsm_compute_returns: io is NULL");
    const int64_t T = io->T, C = io->columns;
    if (T < 0 || C < 0) return fail(2, "lsm_compute_returns: T and columns must be >= 0");
    const bool ptl = io->use_proper_time_limits != 0, gae = io->use_gae != 0;
    const bool denorm = io->value_scale != nullptr;
    if ((io->value_scale == nullptr) != (io->value_shift == nullptr))
        return fail(2, "lsm_compute_returns: value_scale and value_shift are given together or not at all");
    const bool mom = io->stats != nullptr || io->stats64 != nullptr;
    const bool adv = io->advantages != nullptr;
    if (C > 0) {
        if (!io->next_value || !io->returns || (gae && !io->value_preds))
            return fail(2, "lsm_compute_returns: next_value, returns and (GAE) value_preds are required");
        if (T > 0 && (!io->rewards || !io->masks || !io->value_preds || (ptl && !io->bad_masks)))
            return fail(2, "lsm_compute_returns: rewards, masks, value_preds and (proper time limits) bad_masks are required");
    }
    if (mom && (!io->active_masks || !io->scratch))
        return fail(2, "lsm_compute_returns: the advantage moments need active_masks and scratch");
    if (mom && (reinterpret_cast<uintptr_t>(io->scratch) % alignof(double)) != 0)
        return fail(2, "lsm_compute_returns: scratch must be 8-byte aligned");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    int64_t blocks = 0;
    if (C > 0) {
        const int bs = block_threads(C, sm_count());
        blocks = (C + bs - 1) / bs;
        if (blocks > 0x7fffffffLL) return fail(2, "lsm_compute_returns: too many columns");
        ReturnsParams p{T, C, io->rewards, io->value_preds, io->next_value, io->masks, io->bad_masks, io->returns,
                        io->advantages, io->active_masks, io->value_scale, io->value_shift,
                        static_cast<double*>(io->scratch), io->gamma, io->gamma_lambda};
        const int mode = (gae ? 1 : 0) | (ptl ? 2 : 0) | (denorm ? 4 : 0) | (adv ? 8 : 0) | (mom ? 16 : 0);
        kLaunch.f[mode](p, (unsigned)blocks, (unsigned)bs, s);
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return cuda_fail(e, "lsm_returns_kernel");
    }
    if (mom) {
        lsm_returns_moments_kernel<<<1, FINAL_THREADS, 0, s>>>(static_cast<const double*>(io->scratch), blocks,
                                                               io->stats64, io->stats);
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return cuda_fail(e, "lsm_returns_moments_kernel");
    }
    return 0;
}

}  // extern "C"

// lsm_kernels.cu - translation unit of the step kernels for sm_100a.
//
//   lsm_kernel_spec.cuh     kernels specialised at compile time on (dynamics, N, L) - the fast path
//   lsm_kernel_generic.cuh  run-time N / L fallback for every other configuration
//   lsm_step_common.cuh     dynamics, HJ filter resolution, grid interpolation shared by both
//   lsm_filter_op.cuh       the same filter as a standalone batched operator (lsm_safety_filter / lsm_hj_lookup)
//
// Specialised path: three launches per step (per-agent physics -> graph emission -> next step's pair values), see
// lsm_kernel_spec.cuh. Generic path ("warp per env group", one fused launch): a warp owns EPW consecutive
// environments, G = next power of two >= N lanes per environment; per-agent phases run one lane per
// agent; the graph observation is built in the warp's shared-memory slice and written with all 32 lanes.
//
// The reference mutates goal counters / done flags / velocities agent by agent WHILE it emits
// observations (multiagent/environment.py:979-1029). Each agent's own update depends only on its
// own state, so every lane computes its agent's pre- and post-update state in parallel and an
// observer i selects "post" for agents <= i and "pre" for agents > i.
#include "lsm_kernel_generic.cuh"
#include "lsm_kernel_spec.cuh"
#include "lsm_filter_op.cuh"
#include "lsm_edges.cuh"
#include "lsm_rollout.cuh"
#include "lsm_host.h"

#include <climits>
#include <cstdlib>

namespace lsm {

// ---------------------------------------------------------------------------------------------
// host-side launch helpers (used by lsm_capi.cu)
// ---------------------------------------------------------------------------------------------
// (dynamics, N, L, O, warps per env of the emit kernel, resident emit blocks per SM the register budget targets)
#ifndef LSM_AIR_WPE
#define LSM_AIR_WPE 4
#endif
// BASELINE.json's benchmark shapes (8 / 3 / 32 double-integrator agents, 10 airtaxi agents) and the shapes the
// reference's own scripts ship with (train.sh: 4 agents, 2 landmarks, either dynamics; eval_airtaxi.sh: 8 and 16 agents;
// eval_double_integrator.sh: 4 agents; the 16-agent dense golden rollout)
// (dynamics, N, L, O obstacles, ...): O > 0 is the declared obstacle extension (lsm_b200.h num_obstacles) - BASELINE
// configs[2] names "10 airtaxi agents + obstacles", so that shape (4 obstacles) and the bench shape of the double
// integrator with 4 obstacles are specialised too; every other obstacle count runs the generic kernel
#define LSM_SPEC_LIST(X)                               \
    X(LSM_DYN_DOUBLE_INTEGRATOR, 8, 2, 0, 4, 4)        \
    X(LSM_DYN_DOUBLE_INTEGRATOR, 3, 2, 0, 1, 16)       \
    X(LSM_DYN_DOUBLE_INTEGRATOR, 32, 2, 0, 4, 3)       \
    X(LSM_DYN_DOUBLE_INTEGRATOR, 4, 2, 0, 2, 8)        \
    X(LSM_DYN_DOUBLE_INTEGRATOR, 16, 2, 0, 4, 4)       \
    X(LSM_DYN_AIRTAXI, 10, 2, 0, LSM_AIR_WPE, 5)       \
    X(LSM_DYN_AIRTAXI, 4, 2, 0, 2, 8)                  \
    X(LSM_DYN_AIRTAXI, 8, 2, 0, 2, 5)                  \
    X(LSM_DYN_AIRTAXI, 16, 2, 0, 4, 4)                 \
    X(LSM_DYN_AIRTAXI, 10, 2, 4, LSM_AIR_WPE, 5)       \
    X(LSM_DYN_DOUBLE_INTEGRATOR, 8, 2, 4, 4, 4)

// Launch shape of the emit kernel for a shape built on demand (-DLSM_SHAPE below; _build.build_shape), derived
// at compile time instead of measured:
//   WPE   warps per environment. The emit kernel's per-environment phases give one thread per entity or per observer row,
//         so warps beyond ~E / 4 idle; the measured list picks 1 warp at E = 9, 2 at E = 12 and 4 at E = 24 and
//         above, except the 8-agent airtaxi entry (E = 24), measured best at 2.
//   EMINB resident blocks per SM the register budget targets: as many EmitShared blocks as the SM's shared memory holds
//         (1 KB per block reserved by the hardware), at most 512 threads per SM as the list caps it (16 / 8 / 4 blocks
//         of 1 / 2 / 4 warps). E >= ~150 leaves one block per SM.
template <int DYN, int N, int L, int O>
struct ShapeLaunch {
    static constexpr int E = N + N * L + O;
    static constexpr int WPE = E <= 9 ? 1 : E <= 16 ? 2 : 4;
    static constexpr int kSmemPerSm = 233472, kSmemOptin = 232448, kBlockReserved = 1024;
    static constexpr int SMEM = (int)sizeof(EmitShared<DYN, N, L, O, WPE>);
    static_assert(SMEM <= kSmemOptin, "the emit kernel's shared memory exceeds the per-block opt-in of sm_100");
    static constexpr int FIT = kSmemPerSm / (SMEM + kBlockReserved);
    static constexpr int CAP = 16 / WPE;
    static constexpr int EMINB = FIT < 1 ? 1 : FIT > CAP ? CAP : FIT;
};

#ifdef LSM_SHAPE
// a library of exactly one specialised shape (plus the generic kernels). LSM_SHAPE = decimal digits DNNLLOO: dynamics,
// agents, landmarks per agent, obstacles (one integer: nvcc splits a -D value at commas)
constexpr int kShapeDyn = (LSM_SHAPE) / 1000000, kShapeN = (LSM_SHAPE) / 10000 % 100, kShapeL = (LSM_SHAPE) / 100 % 100,
              kShapeO = (LSM_SHAPE) % 100;
static_assert(kShapeDyn == LSM_DYN_DOUBLE_INTEGRATOR || kShapeDyn == LSM_DYN_AIRTAXI, "LSM_SHAPE: dynamics 0 or 1");
using ShapeLaunchT = ShapeLaunch<kShapeDyn, kShapeN, kShapeL, kShapeO>;
#undef LSM_SPEC_LIST
#define LSM_SPEC_LIST(X) X(kShapeDyn, kShapeN, kShapeL, kShapeO, ShapeLaunchT::WPE, ShapeLaunchT::EMINB)
#endif

constexpr int kAgentBlock = 128;
constexpr int kAgentMinB = 2;
constexpr int kPairBlock = kPairThreads;
// SM room the emit grid leaves for pair blocks (placement "late") and the late pair kernel's grid bound. Swept on B200
// with the record-reading pair kernel (profiles/experiments/r03_pair_kernel_sweep.txt, r03_pair_kernel_ab.txt): with no
// room reserved the cfg2 emit kernel gets 6 instead of 5 blocks per SM and ends ~2.5 us earlier; the pair blocks then
// start as emit blocks retire and finish the lookups in the emit kernel's tail (cfg2 -1.1 us against one reserved
// block, cfg4 and cfg5 slightly faster too). A grid bound of 16 blocks per SM lets them fill the SMs the emit kernel frees.
constexpr int kPairResident = 0;
constexpr int kPairLateBlocksPerSm = 16;

// The product library (liblsm_b200.so) has ONE instantiation per kernel and configuration and reads no environment
// variable. Alternative kernel shapes and ablation switches are compiled only with -DLSM_EXPERIMENTS
// (liblsm_b200_exp.so, `_build.build_experiments()`; selected by the tools with LSM_LIB=<path>).
#ifdef LSM_EXPERIMENTS
// LSM_AGENT_MINB=3 trades ~100-400 B of spills for 12 instead of 8 resident physics warps per SM
static int agent_minb() {
    static const int v = [] { const char* e = std::getenv("LSM_AGENT_MINB"); return e ? std::atoi(e) : 0; }();
    return v;
}
static int env_int(const char* name, int dflt) { const char* e = std::getenv(name); return e ? std::atoi(e) : dflt; }
#endif

// The agent and pair kernels exist in two arithmetics of the HJ grid lookups (LSM_FLAG_INTERP_FLOAT32: float32, else
// float64), chosen at compile time; spec_fns picks the pair of the handle's mode. The emit and edge-count kernels make no
// grid lookups and serve both modes.
struct SpecFns {
    const void* pair;         // lsm_pair_kernel for the periodic-dimension mask pair_periodic (kPairPeriodic)
    const void* pair_rt;      // the same kernel reading the mask from the bound grid (any other grid)
    int pair_periodic;
    const void* agent; const void* emit;
    const void* emit_pie;     // emit kernel that also computes the next step's pair values (placement "emit")
    const void* edge_count;   // per-graph edge counts + range prefix for the fused COO output
    int rec_bytes, scratch_bytes, emit_smem, emit_threads;
};

#ifdef LSM_EXPERIMENTS
// LSM_WPE=2|4 selects an alternative emit-kernel shape for the cfg2 specialisation
template <int WPE_, int EMINB_>
static void cfg2_emit_variant(SpecFns* f) {
    f->emit = (const void*)lsm_emit_kernel<LSM_DYN_DOUBLE_INTEGRATOR, 8, 2, 0, WPE_, EMINB_>;
    f->emit_pie = (const void*)lsm_emit_kernel<LSM_DYN_DOUBLE_INTEGRATOR, 8, 2, 0, WPE_, EMINB_, true>;
    f->emit_smem = (int)sizeof(EmitShared<LSM_DYN_DOUBLE_INTEGRATOR, 8, 2, 0, WPE_>);
    f->emit_threads = 32 * WPE_;
}

#endif

static bool spec_fns_base(int dynamics, int N, int L, int O, bool f32, SpecFns* f);
static bool spec_fns(int dynamics, int N, int L, int O, bool f32, SpecFns* f) {
    if (!spec_fns_base(dynamics, N, L, O, f32, f)) return false;
#ifdef LSM_EXPERIMENTS
    if (dynamics == LSM_DYN_DOUBLE_INTEGRATOR && N == 8 && L == 2 && O == 0) {
        const int w = env_int("LSM_WPE", 0);
        if (w == 1) cfg2_emit_variant<1, 8>(f);
        if (w == 2) cfg2_emit_variant<2, 8>(f);
        if (w == 24) cfg2_emit_variant<2, 4>(f);    // two warps per block at half the occupancy target
    }
#endif
    return true;
}

// LSM_AGENT_MINB=3 (lab build) has float64 instantiations only
#ifdef LSM_EXPERIMENTS
#define LSM_AGENT_FN(DYN_, N_, L_, O_, F32_) (agent_minb() == 3 && !(F32_) ? (const void*)lsm_agent_kernel<DYN_, N_, L_, O_, kAgentBlock, 3, false> \
                                                                          : (const void*)lsm_agent_kernel<DYN_, N_, L_, O_, kAgentBlock, kAgentMinB, F32_>)
#define LSM_EMIT_PIE_FN(DYN_, N_, L_, O_, WPE_, EMINB_) ((const void*)lsm_emit_kernel<DYN_, N_, L_, O_, WPE_, EMINB_, true>)
#else
#define LSM_AGENT_FN(DYN_, N_, L_, O_, F32_) ((const void*)lsm_agent_kernel<DYN_, N_, L_, O_, kAgentBlock, kAgentMinB, F32_>)
#define LSM_EMIT_PIE_FN(DYN_, N_, L_, O_, WPE_, EMINB_) nullptr   /* "pair values inside the emit kernel": experiments only */
#endif
static bool spec_fns_base(int dynamics, int N, int L, int O, bool f32, SpecFns* f) {
#define X(DYN_, N_, L_, O_, WPE_, EMINB_)                                                         \
    if (dynamics == DYN_ && N == N_ && L == L_ && O == O_) {                                      \
        f->pair = f32 ? (const void*)lsm_pair_kernel<DYN_, N_, L_, O_, kPairPeriodic<DYN_>, true>  \
                      : (const void*)lsm_pair_kernel<DYN_, N_, L_, O_, kPairPeriodic<DYN_>, false>; \
        f->pair_rt = f32 ? (const void*)lsm_pair_kernel<DYN_, N_, L_, O_, kPeriodicRuntime, true>  \
                         : (const void*)lsm_pair_kernel<DYN_, N_, L_, O_, kPeriodicRuntime, false>; \
        f->pair_periodic = kPairPeriodic<DYN_>;                                                   \
        f->agent = f32 ? LSM_AGENT_FN(DYN_, N_, L_, O_, true) : LSM_AGENT_FN(DYN_, N_, L_, O_, false); \
        f->emit = (const void*)lsm_emit_kernel<DYN_, N_, L_, O_, WPE_, EMINB_>;                   \
        f->emit_pie = LSM_EMIT_PIE_FN(DYN_, N_, L_, O_, WPE_, EMINB_);                            \
        f->edge_count = (const void*)lsm_edge_count_kernel<DYN_, N_, L_, O_>;                     \
        f->rec_bytes = (int)sizeof(EmitRec<DYN_, N_, L_, O_>);                                    \
        f->scratch_bytes = (int)sizeof(AgentScratch<DYN_, N_, L_>);                               \
        f->emit_smem = (int)sizeof(EmitShared<DYN_, N_, L_, O_, WPE_>);                           \
        f->emit_threads = 32 * WPE_;                                                              \
        return true;                                                                              \
    }
    LSM_SPEC_LIST(X)
#undef X
    return false;
}

static const void* generic_ptr(int dynamics) {
    return dynamics == LSM_DYN_DOUBLE_INTEGRATOR ? (const void*)lsm_generic_kernel<LSM_DYN_DOUBLE_INTEGRATOR>
                                                 : (const void*)lsm_generic_kernel<LSM_DYN_AIRTAXI>;
}

static bool kp_interp_f32(const KParams& kp) { return (kp.c.flags & LSM_FLAG_INTERP_FLOAT32) != 0; }

// the geometry is the same in both interpolation modes
bool spec_available(int dynamics, int N, int L, int O, SpecGeometry* g) {
    SpecFns f;
    if (!spec_fns(dynamics, N, L, O, false, &f)) return false;
    g->rec_bytes = f.rec_bytes; g->scratch_bytes = f.scratch_bytes; g->agent_block = kAgentBlock;
    g->emit_smem = f.emit_smem; g->emit_threads = f.emit_threads; g->pair_block = kPairBlock;
    return true;
}

static cudaError_t prepare_one(const void* fn, int block_threads, int smem_bytes, int* regs, int* blocks_per_sm) {
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
    if (e != cudaSuccess) return e;
    cudaFuncAttributes fa;
    e = cudaFuncGetAttributes(&fa, fn);
    if (e != cudaSuccess) return e;
    *regs = fa.numRegs;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, fn, block_threads, smem_bytes);
}

cudaError_t kernel_prepare(int dynamics, int N, int L, int O, bool f32, bool spec, int smem_bytes, int block_threads, int* regs,
                           int* blocks_per_sm) {
    SpecFns f;
    const void* fn = generic_ptr(dynamics);
    if (spec) { if (!spec_fns(dynamics, N, L, O, f32, &f)) return cudaErrorInvalidValue; fn = f.agent; }
    return prepare_one(fn, block_threads, smem_bytes, regs, blocks_per_sm);
}

cudaError_t spec_prepare_aux(int dynamics, int N, int L, int O, bool f32, int* emit_regs, int* emit_blocks_per_sm, int* pair_regs) {
    SpecFns f;
    if (!spec_fns(dynamics, N, L, O, f32, &f)) return cudaErrorInvalidValue;
    cudaError_t e = prepare_one(f.emit, f.emit_threads, f.emit_smem, emit_regs, emit_blocks_per_sm);
    if (e != cudaSuccess) return e;
    if (f.emit_pie != nullptr) { int r = 0, b = 0; e = prepare_one(f.emit_pie, f.emit_threads, f.emit_smem, &r, &b); if (e != cudaSuccess) return e; }
    int bps = 0;
    return prepare_one(f.pair, kPairBlock, 0, pair_regs, &bps);
}

cudaError_t upload_magnetic_tables(const double* cos_tab, const double* sin_tab) {
    cudaError_t e = cudaMemcpyToSymbol(c_mag_cos, cos_tab, sizeof(double) * kMagSegments);
    if (e != cudaSuccess) return e;
    return cudaMemcpyToSymbol(c_mag_sin, sin_tab, sizeof(double) * kMagSegments);
}

static cudaError_t launch_one(const void* fn, const KParams& kp, unsigned grid_blocks, int block_threads, int smem_bytes,
                              cudaStream_t stream, const void* persist_ptr, size_t persist_bytes, bool pdl) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid_blocks, 1, 1);
    cfg.blockDim = dim3((unsigned)block_threads, 1, 1);
    cfg.dynamicSmemBytes = (size_t)smem_bytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    int nattr = 0;
#ifdef LSM_EXPERIMENTS
    static const bool no_pdl = std::getenv("LSM_NO_PDL") != nullptr;
#else
    constexpr bool no_pdl = false;
#endif
    if (pdl && !no_pdl) {
        attr[nattr].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[nattr].val.programmaticStreamSerializationAllowed = 1;
        ++nattr;
    }
    if (persist_ptr != nullptr && persist_bytes > 0) {
        // keep the HJ value grid resident in L2 while the observation stream flows through it
        attr[nattr].id = cudaLaunchAttributeAccessPolicyWindow;
        attr[nattr].val.accessPolicyWindow.base_ptr = const_cast<void*>(persist_ptr);
        attr[nattr].val.accessPolicyWindow.num_bytes = persist_bytes;
        attr[nattr].val.accessPolicyWindow.hitRatio = 1.0f;
        attr[nattr].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        attr[nattr].val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        ++nattr;
    }
    cfg.attrs = attr;
    cfg.numAttrs = nattr;
    void* args[] = { (void*)&kp };
    return cudaLaunchKernelExC(&cfg, fn, args);
}

cudaError_t kernel_launch(const KParams& kp, bool spec, int grid_blocks, int block_threads, int smem_bytes,
                          cudaStream_t stream, const void* persist_ptr, size_t persist_bytes) {
    SpecFns f;
    const void* fn = generic_ptr(kp.c.dynamics);
    if (spec) { if (!spec_fns(kp.c.dynamics, kp.N, kp.L, kp.O, kp_interp_f32(kp), &f)) return cudaErrorInvalidValue; fn = f.agent; }
#ifdef LSM_EXPERIMENTS
    if (spec) {
        // LSM_AGENT_SMEM=<bytes>: pad the agent kernel's dynamic shared memory so that fewer blocks fit an SM and the
        // rest of the SM stays free for emit / pair blocks of another env range (overlap experiment)
        static const int pad = env_int("LSM_AGENT_SMEM", 0);
        if (pad > smem_bytes) {
            static thread_local const void* done = nullptr;
            if (done != fn) { cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, pad); done = fn; }
            smem_bytes = pad;
        }
    }
#endif
    return launch_one(fn, kp, (unsigned)grid_blocks, block_threads, smem_bytes, stream, persist_ptr, persist_bytes, spec);
}

cudaError_t spec_launch_pair(const KParams& kp, cudaStream_t stream, const void* persist_ptr, size_t persist_bytes) {
    SpecFns f;
    if (!spec_fns(kp.c.dynamics, kp.N, kp.L, kp.O, kp_interp_f32(kp), &f)) return cudaErrorInvalidValue;
    // one thread per ordered pair i != j, 32-bit task indices in the kernel
    const long long tasks = (long long)(kp.env_end - kp.env_begin) * kp.N * (kp.N - 1);
    if (tasks > INT_MAX) return cudaErrorInvalidValue;
    int periodic = 0;
    for (int d = 0; d < kp.vg.ndim; ++d) periodic |= kp.vg.periodic[d] ? 1 << d : 0;
    const void* fn = periodic == f.pair_periodic ? f.pair : f.pair_rt;
    long long blocks = (tasks + kPairBlock - 1) / kPairBlock;
    if (blocks < 1) blocks = 1;
    if (kp.pair_late) {
        // beside the emit kernel: a bounded number of resident blocks per SM, each striding over the pairs
        static int sm_count = 0;
        if (sm_count == 0) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev); }
        int bps = kPairLateBlocksPerSm;
#ifdef LSM_EXPERIMENTS
        { const int v = env_int("LSM_PAIR_BPS", 0); if (v >= 1) bps = v; }
#endif
        if (blocks > (long long)sm_count * bps) blocks = (long long)sm_count * bps;
    }
    return launch_one(fn, kp, (unsigned)blocks, kPairBlock, 0, stream, persist_ptr, persist_bytes, true);
}

// resident emit blocks per SM: what fits, minus (when the pair kernel runs beside the emit kernel) enough registers /
// threads for kPairResident pair blocks per SM
static cudaError_t emit_blocks_per_sm(const SpecFns& f, bool reserve_pair, bool pie, int* out) {
    int bps = 0;
    const void* fn = (pie && f.emit_pie != nullptr) ? f.emit_pie : f.emit;
#ifndef LSM_EXPERIMENTS
    // the answer depends only on (kernel, reserve_pair): asked once per process, not on every launch (two occupancy /
    // attribute queries cost more host time than the launch itself)
    struct Memo { const void* fn; const void* pair; bool reserve; int bps; };
    static thread_local Memo memo[32];
    static thread_local int memo_n = 0;
    for (int k = 0; k < memo_n; ++k)
        if (memo[k].fn == fn && memo[k].pair == f.pair && memo[k].reserve == reserve_pair) { *out = memo[k].bps; return cudaSuccess; }
#endif
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, fn, f.emit_threads, f.emit_smem);
    if (e != cudaSuccess) return e;
    if (bps < 1) return cudaErrorLaunchOutOfResources;
    if (reserve_pair) {
        cudaFuncAttributes fe, fp;
        if ((e = cudaFuncGetAttributes(&fe, fn)) != cudaSuccess) return e;
        if ((e = cudaFuncGetAttributes(&fp, f.pair)) != cudaSuccess) return e;
        auto block_regs = [](int regs, int threads) { return ((regs * 32 + 255) / 256 * 256) * ((threads + 31) / 32); };
        int resident = kPairResident;
#ifdef LSM_EXPERIMENTS
        { const int v = env_int("LSM_PAIR_RESIDENT", -1); if (v >= 0) resident = v; }
#endif
        const int need_regs = resident * block_regs(fp.numRegs, kPairBlock), need_thr = resident * kPairBlock;
        while (bps > 1 && (65536 - bps * block_regs(fe.numRegs, f.emit_threads) < need_regs || 2048 - bps * f.emit_threads < need_thr)) --bps;
    }
#ifdef LSM_EXPERIMENTS
    { const int v = env_int("LSM_EMIT_BPS", 0); if (v >= 1 && v < bps) bps = v; }
#else
    if (memo_n < 32) { memo[memo_n].fn = fn; memo[memo_n].pair = f.pair; memo[memo_n].reserve = reserve_pair; memo[memo_n].bps = bps; ++memo_n; }
#endif
    *out = bps;
    return cudaSuccess;
}

cudaError_t spec_emit_blocks_per_sm(int dynamics, int N, int L, int O, bool f32, bool reserve_pair, bool pie, int* out, int* regs) {
    SpecFns f;
    if (!spec_fns(dynamics, N, L, O, f32, &f)) return cudaErrorInvalidValue;
    if (regs != nullptr) {
        cudaFuncAttributes fa;
        cudaError_t e = cudaFuncGetAttributes(&fa, (pie && f.emit_pie != nullptr) ? f.emit_pie : f.emit);
        if (e != cudaSuccess) return e;
        *regs = fa.numRegs;
    }
    return emit_blocks_per_sm(f, reserve_pair, pie, out);
}

cudaError_t spec_launch_emit(const KParams& kp, cudaStream_t stream, const void* persist_ptr, size_t persist_bytes, bool reserve_pair, bool pie) {
    SpecFns f;
    if (!spec_fns(kp.c.dynamics, kp.N, kp.L, kp.O, kp_interp_f32(kp), &f)) return cudaErrorInvalidValue;
    // persistent blocks: as many as are resident at once, each loops over environments
    static int sm_count = 0;
    if (sm_count == 0) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev); }
    int bps = 0;
    cudaError_t e = emit_blocks_per_sm(f, reserve_pair, pie, &bps);
    if (e != cudaSuccess) return e;
    unsigned grid = (unsigned)sm_count * (unsigned)bps;
    if (grid > (unsigned)(kp.env_end - kp.env_begin)) grid = (unsigned)(kp.env_end - kp.env_begin);
    if (grid < 1) grid = 1;
#ifdef LSM_EXPERIMENTS
    { const unsigned v = (unsigned)env_int("LSM_EMIT_GRID", 0); if (v >= 1 && v < grid) grid = v; }
#endif
    if (pie && f.emit_pie == nullptr) return cudaErrorInvalidValue;
    return launch_one(pie ? f.emit_pie : f.emit, kp, grid, f.emit_threads, f.emit_smem, stream, persist_ptr, persist_bytes, true);
}

int edge_count_envs_per_block(long long envs) {
    // contiguous env runs per block: at least one env per warp, at most ~2048 blocks, at most kEdgeMaxEnvsPerBlock
    long long c = (envs + 2047) / 2048;
    if (c < kEdgeCountWarps) c = kEdgeCountWarps;
    if (c > kEdgeMaxEnvsPerBlock) c = kEdgeMaxEnvsPerBlock;
    return (int)c;
}

cudaError_t spec_launch_edge_count(const KParams& kp, cudaStream_t stream) {
    SpecFns f;
    if (!spec_fns(kp.c.dynamics, kp.N, kp.L, kp.O, kp_interp_f32(kp), &f)) return cudaErrorInvalidValue;
    const long long envs = kp.env_end - kp.env_begin;
    long long blocks = (envs + kp.edge_envs_per_block - 1) / kp.edge_envs_per_block;
    if (blocks < 1) blocks = 1;
    return launch_one(f.edge_count, kp, (unsigned)blocks, 32 * kEdgeCountWarps, 0, stream, nullptr, 0, true);
}

cudaError_t world_graph_launch(const KParams& kp, int32_t* counts, long long* offsets, long long* edge_index, double* edge_weight,
                               long long capacity, cudaStream_t stream) {
    const int wpb = 4;
    const unsigned blocks = (unsigned)((kp.b.num_envs + wpb - 1) / wpb);
    lsm_world_graph_kernel<<<blocks, wpb * 32, 0, stream>>>(kp, 0, counts, offsets, edge_index, edge_weight, capacity);
    lsm_edge_scan_kernel<<<1, 1024, 0, stream>>>(counts, offsets, kp.b.num_envs);
    lsm_world_graph_kernel<<<blocks, wpb * 32, 0, stream>>>(kp, 1, counts, offsets, edge_index, edge_weight, capacity);
    return cudaGetLastError();
}

cudaError_t pack_grid_launch(const GridDev& g, float* packed, long long cells) {
    const long long total = cells << g.ndim;
    const unsigned blocks = (unsigned)((total + 255) / 256);
    if (g.ndim == 4) lsm_pack_grid_kernel<4><<<blocks, 256>>>(g.values, packed, g, cells);
    else if (g.ndim == 5) lsm_pack_grid_kernel<5><<<blocks, 256>>>(g.values, packed, g, cells);
    else return cudaErrorInvalidValue;
    return cudaGetLastError();
}

cudaError_t episode_stats_launch(const double* ep_info, long long n, double* out, cudaStream_t stream) {
    lsm_episode_stats_kernel<<<1, 256, 0, stream>>>(ep_info, n, LSM_EP_COUNT, out);
    return cudaGetLastError();
}

cudaError_t rollout_insert_launch(const float* obs, const uint8_t* done, float* share_obs, float* masks, float* active_masks,
                                  long long n, int N, int D, cudaStream_t stream) {
    const long long total = n * (long long)N * N * D;
    long long blocks = (total + 255) / 256;
    if (blocks > 148LL * 16) blocks = 148LL * 16;
    lsm_rollout_insert_kernel<<<(unsigned)blocks, 256, 0, stream>>>(obs, done, share_obs, masks, active_masks, n, N, D);
    return cudaGetLastError();
}

// include/lsm_math.h evaluated on the device (bit-identity test against the host / oracle evaluation)
__global__ void __launch_bounds__(256) lsm_math_eval_kernel(int op, const double* __restrict__ a, const double* __restrict__ b,
                                                          double* __restrict__ out, long long n) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    if (op == 0) out[k] = lsm_sin(a[k]);
    else if (op == 1) out[k] = lsm_cos(a[k]);
    else if (op == 2) out[k] = lsm_atan2(a[k], b[k]);
    else { double s, c; lsm_sincos(a[k], &s, &c); out[k] = (op == 3) ? s : c; }
}
cudaError_t math_eval_launch(int op, const double* a, const double* b, double* out, long long n, cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    lsm_math_eval_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(op, a, b, out, n);
    return cudaGetLastError();
}

// the standalone filter operator: instantiation of the handle's dynamics and interpolation mode, on the caller's stream
static int sm_count_cached() {
    static int sm_count = 0;
    if (sm_count == 0) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev); }
    return sm_count;
}

cudaError_t safety_filter_launch(const KParams& kp, const FilterOpArgs& a, cudaStream_t stream) {
    if (a.rows <= 0) return cudaSuccess;
    const bool f32 = kp_interp_f32(kp), di = kp.c.dynamics == LSM_DYN_DOUBLE_INTEGRATOR;
    const void* fn = di ? (f32 ? (const void*)lsm_safety_filter_kernel<LSM_DYN_DOUBLE_INTEGRATOR, true>
                               : (const void*)lsm_safety_filter_kernel<LSM_DYN_DOUBLE_INTEGRATOR, false>)
                        : (f32 ? (const void*)lsm_safety_filter_kernel<LSM_DYN_AIRTAXI, true>
                               : (const void*)lsm_safety_filter_kernel<LSM_DYN_AIRTAXI, false>);
    // one tile of kFopRows rows per block; beyond 32 blocks per SM the blocks stride over the tiles
    long long blocks = (a.rows + kFopRows - 1) / kFopRows;
    const long long cap = (long long)sm_count_cached() * 32;
    if (blocks > cap) blocks = cap;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)blocks, 1, 1);
    cfg.blockDim = dim3(kFopThreads, 1, 1);
    cfg.stream = stream;
    void* args[] = { (void*)&kp, (void*)&a };
    return cudaLaunchKernelExC(&cfg, fn, args);
}

cudaError_t hj_lookup_launch(const KParams& kp, const LookupArgs& a, cudaStream_t stream) {
    if (a.points <= 0) return cudaSuccess;
    const bool f32 = kp_interp_f32(kp), di = kp.c.dynamics == LSM_DYN_DOUBLE_INTEGRATOR;
    const void* fn = di ? (f32 ? (const void*)lsm_hj_lookup_kernel<LSM_DYN_DOUBLE_INTEGRATOR, true>
                               : (const void*)lsm_hj_lookup_kernel<LSM_DYN_DOUBLE_INTEGRATOR, false>)
                        : (f32 ? (const void*)lsm_hj_lookup_kernel<LSM_DYN_AIRTAXI, true>
                               : (const void*)lsm_hj_lookup_kernel<LSM_DYN_AIRTAXI, false>);
    long long blocks = (a.points + kLookupThreads - 1) / kLookupThreads;
    const long long cap = (long long)sm_count_cached() * 64;
    if (blocks > cap) blocks = cap;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)blocks, 1, 1);
    cfg.blockDim = dim3(kLookupThreads, 1, 1);
    cfg.stream = stream;
    void* args[] = { (void*)&kp, (void*)&a };
    return cudaLaunchKernelExC(&cfg, fn, args);
}

cudaError_t pad_grads_launch(const float* grads, float* grads8, long long cells) {
    lsm_pad_grads_kernel<<<(unsigned)((cells * 8 + 255) / 256), 256>>>(grads, grads8, cells);
    return cudaGetLastError();
}

cudaError_t edge_list_launch(const float* adj, int32_t* counts, long long* offsets, long long* edge_index, float* edge_attr,
                             long long num_graphs, int E, long long capacity, cudaStream_t stream) {
    const int wpb = 8;   // warps (graphs) per block
    const unsigned blocks = (unsigned)((num_graphs + wpb - 1) / wpb);
    lsm_edge_count_kernel<<<blocks, wpb * 32, 0, stream>>>(adj, counts, num_graphs, E * E);
    lsm_edge_scan_kernel<<<1, 1024, 0, stream>>>(counts, offsets, num_graphs);
    lsm_edge_fill_kernel<<<blocks, wpb * 32, 0, stream>>>(adj, offsets, edge_index, edge_attr, num_graphs, E, capacity);
    return cudaGetLastError();
}

}  // namespace lsm

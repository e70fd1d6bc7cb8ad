// lsm_kernels.cu - translation unit of the step kernels for sm_100a.
//
//   lsm_kernel_spec.cuh     kernels specialised at compile time on (dynamics, N, L) - the fast path
//   lsm_kernel_generic.cuh  run-time N / L fallback for every other configuration
//   lsm_step_common.cuh     dynamics and HJ filter resolution shared by both
//   lsm_grid.cuh            the HJ grid lookups of every kernel, in both arithmetics, and the grid-copy builders
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

namespace lsm {

// ---------------------------------------------------------------------------------------------
// host-side launch helpers (used by lsm_capi.cu)
// ---------------------------------------------------------------------------------------------
// (dynamics, N, L, O, warps per env of the emit kernel, resident emit blocks per SM the register budget targets)
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
    X(LSM_DYN_AIRTAXI, 10, 2, 0, 4, 5)                 \
    X(LSM_DYN_AIRTAXI, 4, 2, 0, 2, 8)                  \
    X(LSM_DYN_AIRTAXI, 8, 2, 0, 2, 5)                  \
    X(LSM_DYN_AIRTAXI, 16, 2, 0, 4, 4)                 \
    X(LSM_DYN_AIRTAXI, 10, 2, 4, 4, 5)                 \
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
// Grid bound of the late pair kernel (placement 0). Swept on B200 with the record-reading pair kernel
// (profiles/experiments/r03_pair_kernel_sweep.txt, r03_pair_kernel_ab.txt): the emit grid reserves no room for pair
// blocks; they start as emit blocks retire and finish the lookups in the emit kernel's tail, and 16 blocks per SM lets
// them fill the SMs the emit kernel frees.
constexpr int kPairLateBlocksPerSm = 16;

// The agent and pair kernels exist in two arithmetics of the HJ grid lookups (LSM_FLAG_INTERP_FLOAT32: float32, else
// float64), chosen at compile time; the table holds the pair of the handle's mode. The emit, edge-count and record
// kernels make no grid lookups and serve both modes.
bool spec_table(int dynamics, int N, int L, int O, bool f32, SpecTable* t) {
    *t = SpecTable{};
#define X(DYN_, N_, L_, O_, WPE_, EMINB_)                                                         \
    if (dynamics == DYN_ && N == N_ && L == L_ && O == O_) {                                      \
        t->agent = f32 ? (const void*)lsm_agent_kernel<DYN_, N_, L_, O_, kAgentBlock, kAgentMinB, true>  \
                       : (const void*)lsm_agent_kernel<DYN_, N_, L_, O_, kAgentBlock, kAgentMinB, false>; \
        t->pair = f32 ? (const void*)lsm_pair_kernel<DYN_, N_, L_, O_, kPairPeriodic<DYN_>, true>  \
                      : (const void*)lsm_pair_kernel<DYN_, N_, L_, O_, kPairPeriodic<DYN_>, false>; \
        t->pair_rt = f32 ? (const void*)lsm_pair_kernel<DYN_, N_, L_, O_, kPeriodicRuntime, true>  \
                         : (const void*)lsm_pair_kernel<DYN_, N_, L_, O_, kPeriodicRuntime, false>; \
        t->pair_periodic = kPairPeriodic<DYN_>;                                                   \
        t->emit = (const void*)lsm_emit_kernel<DYN_, N_, L_, O_, WPE_, EMINB_>;                   \
        t->edge_count = (const void*)lsm_edge_count_kernel<DYN_, N_, L_, O_>;                     \
        t->rec_bytes = (int)sizeof(EmitRec<DYN_, N_, L_, O_>);                                    \
        t->scratch_bytes = (int)sizeof(AgentScratch<DYN_, N_, L_>);                               \
        t->agent_block = kAgentBlock;                                                             \
        t->emit_smem = (int)sizeof(EmitShared<DYN_, N_, L_, O_, WPE_>);                           \
        t->emit_threads = 32 * WPE_;                                                              \
        t->record_emit = (const void*)lsm_record_emit_kernel<DYN_, N_, L_, O_>;                   \
        t->record_emit_smem = RecordEmitGeom<DYN_, N_, L_, O_>::SMEM;                             \
        t->record_emit_threads = RecordEmitGeom<DYN_, N_, L_, O_>::THREADS;                       \
        t->record_emit_items = RecordEmitGeom<DYN_, N_, L_, O_>::GPB;                             \
        t->record_edge_count = (const void*)lsm_record_emit_kernel_edge_count<DYN_, N_, L_, O_>;  \
        t->record_edge_fill = (const void*)lsm_record_emit_kernel_edge_fill<DYN_, N_, L_, O_>;    \
        t->record_edges_smem = RecordEdgesGeom<DYN_, N_, L_, O_>::SMEM;                           \
        t->record_edges_threads = RecordEdgesGeom<DYN_, N_, L_, O_>::THREADS;                     \
        t->record_edges_items = RecordEdgesGeom<DYN_, N_, L_, O_>::GPB;                           \
        return true;                                                                              \
    }
    LSM_SPEC_LIST(X)
#undef X
    return false;
}

const void* generic_ptr(int dynamics) {
    return dynamics == LSM_DYN_DOUBLE_INTEGRATOR ? (const void*)lsm_generic_kernel<LSM_DYN_DOUBLE_INTEGRATOR>
                                                 : (const void*)lsm_generic_kernel<LSM_DYN_AIRTAXI>;
}

static bool kp_float32_lookups(const KParams& kp) { return (kp.c.flags & LSM_FLAG_INTERP_FLOAT32) != 0; }

cudaError_t kernel_prepare(const void* fn, int block_threads, int smem_bytes, int* regs, int* blocks_per_sm) {
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
    if (e != cudaSuccess) return e;
    cudaFuncAttributes fa;
    e = cudaFuncGetAttributes(&fa, fn);
    if (e != cudaSuccess) return e;
    *regs = fa.numRegs;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, fn, block_threads, smem_bytes);
}

cudaError_t spec_prepare(SpecTable* t) {
    cudaError_t e = kernel_prepare(t->emit, t->emit_threads, t->emit_smem, &t->emit_regs, &t->emit_blocks_per_sm);
    if (e != cudaSuccess) return e;
    int bps = 0;
    return kernel_prepare(t->pair, kPairBlock, 0, &t->pair_regs, &bps);
}

cudaError_t upload_magnetic_tables(const double* cos_tab, const double* sin_tab) {
    cudaError_t e = cudaMemcpyToSymbol(c_mag_cos, cos_tab, sizeof(double) * kMagSegments);
    if (e != cudaSuccess) return e;
    return cudaMemcpyToSymbol(c_mag_sin, sin_tab, sizeof(double) * kMagSegments);
}

cudaError_t kernel_launch(const void* fn, const KParams& kp, unsigned grid_blocks, int block_threads, int smem_bytes,
                          cudaStream_t stream, bool pdl) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid_blocks, 1, 1);
    cfg.blockDim = dim3((unsigned)block_threads, 1, 1);
    cfg.dynamicSmemBytes = (size_t)smem_bytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    int nattr = 0;
    if (pdl) {
        attr[nattr].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[nattr].val.programmaticStreamSerializationAllowed = 1;
        ++nattr;
    }
    cfg.attrs = attr;
    cfg.numAttrs = nattr;
    void* args[] = { (void*)&kp };
    return cudaLaunchKernelExC(&cfg, fn, args);
}

cudaError_t spec_launch_pair(const KParams& kp, const SpecTable& t, int sm_count, cudaStream_t stream) {
    // one thread per ordered pair i != j, 32-bit task indices in the kernel
    const long long tasks = (long long)(kp.env_end - kp.env_begin) * kp.N * (kp.N - 1);
    if (tasks > INT_MAX) return cudaErrorInvalidValue;
    int periodic = 0;
    for (int d = 0; d < kp.vg.ndim; ++d) periodic |= kp.vg.periodic[d] ? 1 << d : 0;
    const void* fn = periodic == t.pair_periodic ? t.pair : t.pair_rt;
    long long blocks = (tasks + kPairBlock - 1) / kPairBlock;
    if (blocks < 1) blocks = 1;
    // beside the emit kernel: a bounded number of resident blocks per SM, each striding over the pairs
    if (kp.pair_late && blocks > (long long)sm_count * kPairLateBlocksPerSm) blocks = (long long)sm_count * kPairLateBlocksPerSm;
    return kernel_launch(fn, kp, (unsigned)blocks, kPairBlock, 0, stream, true);
}

cudaError_t spec_launch_emit(const KParams& kp, const SpecTable& t, int sm_count, cudaStream_t stream) {
    // persistent blocks: as many as are resident at once, each loops over environments
    unsigned grid = (unsigned)sm_count * (unsigned)t.emit_blocks_per_sm;
    if (grid > (unsigned)(kp.env_end - kp.env_begin)) grid = (unsigned)(kp.env_end - kp.env_begin);
    if (grid < 1) grid = 1;
    return kernel_launch(t.emit, kp, grid, t.emit_threads, t.emit_smem, stream, true);
}

cudaError_t spec_launch_record_emit(const SpecTable& t, int sm_count, const RecordEmitArgs& a, cudaStream_t stream) {
    if (a.num_items <= 0) return cudaSuccess;
    if (t.record_emit_smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(t.record_emit, cudaFuncAttributeMaxDynamicSharedMemorySize, t.record_emit_smem);
        if (e != cudaSuccess) return e;
    }
    // blocks loop over the items: at most as many as 8 blocks of 256 threads per SM (a full SM) hold
    long long blocks = (a.num_items + t.record_emit_items - 1) / t.record_emit_items;
    if (blocks > 8LL * sm_count) blocks = 8LL * sm_count;
    void* args[] = { (void*)&a };
    return cudaLaunchKernel(t.record_emit, dim3((unsigned)blocks), dim3((unsigned)t.record_emit_threads), args,
                            (size_t)t.record_emit_smem, stream);
}

cudaError_t spec_launch_record_edges(const SpecTable& t, int sm_count, const RecordEdgesArgs& a, long long* offsets, bool fill,
                                     cudaStream_t stream) {
    if (a.num_items <= 0) return fill ? cudaSuccess : cudaMemsetAsync(offsets, 0, sizeof(long long), stream);
    const void* fn = fill ? t.record_edge_fill : t.record_edge_count;
    if (t.record_edges_smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, t.record_edges_smem);
        if (e != cudaSuccess) return e;
    }
    // blocks loop over the items, as in spec_launch_record_emit
    long long blocks = (a.num_items + t.record_edges_items - 1) / t.record_edges_items;
    if (blocks > 8LL * sm_count) blocks = 8LL * sm_count;
    void* args[] = { (void*)&a };
    cudaError_t e = cudaLaunchKernel(fn, dim3((unsigned)blocks), dim3((unsigned)t.record_edges_threads), args,
                                     (size_t)t.record_edges_smem, stream);
    if (e != cudaSuccess || fill) return e;
    lsm_edge_scan_kernel<<<1, 1024, 0, stream>>>(a.counts, offsets, a.num_items);
    return cudaGetLastError();
}

int edge_count_envs_per_block(long long envs) {
    // contiguous env runs per block: at least one env per warp, at most ~2048 blocks, at most kEdgeMaxEnvsPerBlock
    long long c = (envs + 2047) / 2048;
    if (c < kEdgeCountWarps) c = kEdgeCountWarps;
    if (c > kEdgeMaxEnvsPerBlock) c = kEdgeMaxEnvsPerBlock;
    return (int)c;
}

cudaError_t spec_launch_edge_count(const KParams& kp, const SpecTable& t, cudaStream_t stream) {
    const long long envs = kp.env_end - kp.env_begin;
    long long blocks = (envs + kp.edge_envs_per_block - 1) / kp.edge_envs_per_block;
    if (blocks < 1) blocks = 1;
    return kernel_launch(t.edge_count, kp, (unsigned)blocks, 32 * kEdgeCountWarps, 0, stream, true);
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
cudaError_t safety_filter_launch(const KParams& kp, int sm_count, const FilterOpArgs& a, cudaStream_t stream) {
    if (a.rows <= 0) return cudaSuccess;
    const bool f32 = kp_float32_lookups(kp), di = kp.c.dynamics == LSM_DYN_DOUBLE_INTEGRATOR;
    const void* fn = di ? (f32 ? (const void*)lsm_safety_filter_kernel<LSM_DYN_DOUBLE_INTEGRATOR, true>
                               : (const void*)lsm_safety_filter_kernel<LSM_DYN_DOUBLE_INTEGRATOR, false>)
                        : (f32 ? (const void*)lsm_safety_filter_kernel<LSM_DYN_AIRTAXI, true>
                               : (const void*)lsm_safety_filter_kernel<LSM_DYN_AIRTAXI, false>);
    // one tile of kFopRows rows per block; beyond 32 blocks per SM the blocks stride over the tiles
    long long blocks = (a.rows + kFopRows - 1) / kFopRows;
    const long long cap = (long long)sm_count * 32;
    if (blocks > cap) blocks = cap;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)blocks, 1, 1);
    cfg.blockDim = dim3(kFopThreads, 1, 1);
    cfg.stream = stream;
    void* args[] = { (void*)&kp, (void*)&a };
    return cudaLaunchKernelExC(&cfg, fn, args);
}

cudaError_t hj_lookup_launch(const KParams& kp, int sm_count, const LookupArgs& a, cudaStream_t stream) {
    if (a.points <= 0) return cudaSuccess;
    const bool f32 = kp_float32_lookups(kp), di = kp.c.dynamics == LSM_DYN_DOUBLE_INTEGRATOR;
    const void* fn = di ? (f32 ? (const void*)lsm_hj_lookup_kernel<LSM_DYN_DOUBLE_INTEGRATOR, true>
                               : (const void*)lsm_hj_lookup_kernel<LSM_DYN_DOUBLE_INTEGRATOR, false>)
                        : (f32 ? (const void*)lsm_hj_lookup_kernel<LSM_DYN_AIRTAXI, true>
                               : (const void*)lsm_hj_lookup_kernel<LSM_DYN_AIRTAXI, false>);
    long long blocks = (a.points + kLookupThreads - 1) / kLookupThreads;
    const long long cap = (long long)sm_count * 64;
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

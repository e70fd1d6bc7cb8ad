// lsm_host.h - host-visible launch helpers implemented next to the kernels (lsm_kernels.cu).
#pragma once
#include "lsm_device.cuh"

namespace lsm {
// The kernels and launch geometry of one specialised shape in one interpolation mode: lsm_create fills it once per handle
// (spec_table, then spec_prepare) and every launcher of the specialised pipeline reads it.
struct SpecTable {
    const void* agent;        // lsm_agent_kernel
    const void* pair;         // lsm_pair_kernel for the periodic-dimension mask pair_periodic (kPairPeriodic)
    const void* pair_rt;      // the same kernel reading the mask from the bound grid (any other grid)
    int pair_periodic;
    const void* emit;
    const void* edge_count;   // per-graph edge counts + range prefix for the fused COO output
    int rec_bytes;            // sizeof(EmitRec): per-env record between the agent and the emit kernel
    int scratch_bytes;        // sizeof(AgentScratch): per-env physics scratch of the agent kernel
    int agent_block;
    int emit_smem, emit_threads;
    int emit_regs, emit_blocks_per_sm, pair_regs;   // spec_prepare
    const void* record_emit;  // lsm_record_emit_kernel (lsm_emit_from_records)
    int record_emit_smem, record_emit_threads, record_emit_items;   // items in flight per block
    const void* record_edge_count;  // lsm_record_emit_kernel_edge_count / _edge_fill (lsm_edges_from_records)
    const void* record_edge_fill;
    int record_edges_smem, record_edges_threads, record_edges_items;
};
// the table of (dynamics, N, L, O) with the agent / pair kernels of the interpolation mode (f32: LSM_FLAG_INTERP_FLOAT32);
// false (table zeroed): no specialisation, the shape runs the fused generic kernel
bool spec_table(int dynamics, int N, int L, int O, bool f32, SpecTable* t);
// dynamic shared memory opt-in of the emit kernel, its registers and resident blocks per SM, the pair kernel's registers
cudaError_t spec_prepare(SpecTable* t);
const void* generic_ptr(int dynamics);
// dynamic shared memory opt-in of `fn`, its registers and resident blocks per SM
cudaError_t kernel_prepare(const void* fn, int block_threads, int smem_bytes, int* regs, int* blocks_per_sm);
cudaError_t upload_magnetic_tables(const double* cos_tab, const double* sin_tab);
// one kernel taking the KParams block; pdl: programmatic stream serialisation with the launch before it
cudaError_t kernel_launch(const void* fn, const KParams& kp, unsigned grid_blocks, int block_threads, int smem_bytes,
                          cudaStream_t stream, bool pdl);
cudaError_t spec_launch_pair(const KParams& kp, const SpecTable& t, int sm_count, cudaStream_t stream);
cudaError_t spec_launch_emit(const KParams& kp, const SpecTable& t, int sm_count, cudaStream_t stream);
// lsm_record_emit_kernel of the shape; no-op for zero items
cudaError_t spec_launch_record_emit(const SpecTable& t, int sm_count, const RecordEmitArgs& a, cudaStream_t stream);
// lsm_record_emit_kernel_edge_count + lsm_edge_scan_kernel into `offsets` (fill == false), or
// lsm_record_emit_kernel_edge_fill (fill == true); zero items: the count pass only sets offsets[0] = 0
cudaError_t spec_launch_record_edges(const SpecTable& t, int sm_count, const RecordEdgesArgs& a, long long* offsets, bool fill,
                                     cudaStream_t stream);
int edge_count_envs_per_block(long long envs);
cudaError_t spec_launch_edge_count(const KParams& kp, const SpecTable& t, cudaStream_t stream);
cudaError_t world_graph_launch(const KParams& kp, int32_t* counts, long long* offsets, long long* edge_index, double* edge_weight,
                               long long capacity, cudaStream_t stream);
cudaError_t pack_grid_launch(const GridDev& g, float* packed, long long cells);
cudaError_t episode_stats_launch(const double* ep_info, long long n, double* out, cudaStream_t stream);
cudaError_t rollout_insert_launch(const float* obs, const uint8_t* done, float* share_obs, float* masks, float* active_masks,
                                  long long n, int N, int D, cudaStream_t stream);
cudaError_t math_eval_launch(int op, const double* a, const double* b, double* out, long long n, cudaStream_t stream);
// standalone filter operator (lsm_filter_op.cuh): device pointers of lsm_filter_io / lsm_lookup_io
struct FilterOpArgs {
    long long rows;
    int slots;
    const double* ego;              // [rows][4]
    const double* others;           // [rows][slots][4]
    const double* ego_action;       // [rows][2]
    const double* other_actions;    // [rows][slots][2]
    const uint8_t* active;          // [rows][slots] or NULL (all active)
    const double* sep;              // [rows] or NULL (the grid's own separation: no shift)
    double* safe_action;            // [rows][2]
    uint8_t* filtered;              // [rows] or NULL
    int32_t* index;                 // [rows] or NULL
    double* value;                  // [rows] or NULL
};

struct LookupArgs {
    long long points;
    const double* rel;              // [points][ND] or NULL: then (ego, other) pairs
    const double* ego;              // [points][4]
    const double* other;            // [points][4]
    const double* sep;              // [points] or NULL
    double* value;                  // [points]
    double* grad;                   // [points][ND] or NULL
    double* rel_out;                // [points][ND] or NULL
};
// lsm_filter_op.cuh: the handle's dynamics and interpolation mode; no-op for zero rows / points
cudaError_t safety_filter_launch(const KParams& kp, int sm_count, const FilterOpArgs& a, cudaStream_t stream);
cudaError_t hj_lookup_launch(const KParams& kp, int sm_count, const LookupArgs& a, cudaStream_t stream);
cudaError_t pad_grads_launch(const float* grads, float* grads8, long long cells);
cudaError_t edge_list_launch(const float* adj, int32_t* counts, long long* offsets, long long* edge_index, float* edge_attr,
                             long long num_graphs, int E, long long capacity, cudaStream_t stream);
}  // namespace lsm

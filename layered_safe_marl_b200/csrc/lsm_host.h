// lsm_host.h - host-visible launch helpers implemented next to the kernels (lsm_kernels.cu).
#pragma once
#include "lsm_device.cuh"

namespace lsm {
struct SpecGeometry {
    int rec_bytes;        // sizeof(EmitRec): per-env record between the agent and the emit kernel
    int scratch_bytes;    // sizeof(AgentScratch): per-env physics scratch of the agent kernel
    int agent_block, pair_block;
    int emit_smem, emit_threads;
};
bool spec_available(int dynamics, int N, int L, int O, SpecGeometry* g);
// agent kernel (specialised) or the fused generic kernel
// f32: the LSM_FLAG_INTERP_FLOAT32 instantiations of the agent / pair kernels (specialised path)
cudaError_t kernel_prepare(int dynamics, int N, int L, int O, bool f32, bool spec, int smem_bytes, int block_threads, int* regs,
                           int* blocks_per_sm);
cudaError_t spec_prepare_aux(int dynamics, int N, int L, int O, bool f32, int* emit_regs, int* emit_blocks_per_sm, int* pair_regs);
cudaError_t upload_magnetic_tables(const double* cos_tab, const double* sin_tab);
cudaError_t kernel_launch(const KParams& kp, bool spec, int grid_blocks, int block_threads, int smem_bytes,
                          cudaStream_t stream, const void* persist_ptr, size_t persist_bytes);
cudaError_t spec_launch_pair(const KParams& kp, cudaStream_t stream, const void* persist_ptr, size_t persist_bytes);
cudaError_t spec_launch_emit(const KParams& kp, cudaStream_t stream, const void* persist_ptr, size_t persist_bytes, bool reserve_pair, bool pie);
cudaError_t spec_emit_blocks_per_sm(int dynamics, int N, int L, int O, bool f32, bool reserve_pair, bool pie, int* out, int* regs);
int edge_count_envs_per_block(long long envs);
cudaError_t spec_launch_edge_count(const KParams& kp, cudaStream_t stream);
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
cudaError_t safety_filter_launch(const KParams& kp, const FilterOpArgs& a, cudaStream_t stream);
cudaError_t hj_lookup_launch(const KParams& kp, const LookupArgs& a, cudaStream_t stream);
cudaError_t pad_grads_launch(const float* grads, float* grads8, long long cells);
cudaError_t edge_list_launch(const float* adj, int32_t* counts, long long* offsets, long long* edge_index, float* edge_attr,
                             long long num_graphs, int E, long long capacity, cudaStream_t stream);
}  // namespace lsm

// lsm_edges.cuh - compacted COO edge list of the step's adjacency output, in the order the policy's GNN expects
// (SURVEY.md section 8f, row N2).
//
// Replaces `TransformerConvNet.process_adj` (reference onpolicy/algorithms/utils/gnn.py:376-407), which runs on every
// policy forward: adj (B, E, E) -> adj.nonzero() in row-major (graph, row, col) order ->
//     edge_index = [graph * E + row, graph * E + col]   (2, nnz) int64
//     edge_attr  = adj[graph, row, col]                  (nnz, 1) float32
// with B = num_envs * N graphs (the runner concatenates the agent axis into the batch, graph_mpe_runner.py:398-410).
//
// Three ways to get it. (1) lsm_set_edge_output: the step pipeline itself writes the list (lsm_edge_count_kernel<DYN,N,L>
// below + the edge section of lsm_emit_kernel), the dense adjacency becomes optional and nothing is read back.
// (2) lsm_edge_list: a post-pass over ANY dense adjacency tensor (a rollout-buffer slot, a user tensor) -
// three launches, all HBM / L2 streaming integer work (no tensor cores):
//   lsm_edge_count_kernel   one warp per graph: popcount of the non-zero entries -> counts[g]
//   lsm_edge_scan_kernel    one block: exclusive prefix sum of counts -> offsets[g], offsets[B] = nnz
//   lsm_edge_fill_kernel    one warp per graph: row-major walk in chunks of 32 entries, ballot + prefix popcount
//                           compaction, writes starting at offsets[g]
// The dense matrices are read twice; they were just written by the emit kernel and mostly sit in the 126 MB L2.
// (3) lsm_edges_from_records: the list of (stored record, observer) items of a rollout store - a learner minibatch -
// computed from the records like (1), with no dense matrix (lsm_record_emit_kernel_edge_count / _edge_fill in
// lsm_kernel_spec.cuh, lsm_edge_scan_kernel between them).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace lsm {

__global__ void __launch_bounds__(256) lsm_edge_count_kernel(const float* __restrict__ adj, int32_t* __restrict__ counts,
                                                             long long num_graphs, int EE) {
    const long long g = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (g >= num_graphs) return;
    const int lane = threadIdx.x & 31;
    const float* a = adj + g * EE;
    int c = 0;
    if ((EE & 3) == 0 && ((reinterpret_cast<uintptr_t>(a) & 15u) == 0)) {
        const float4* a4 = reinterpret_cast<const float4*>(a);
        for (int k = lane; k < EE / 4; k += 32) {
            const float4 v = a4[k];
            c += (v.x != 0.0f) + (v.y != 0.0f) + (v.z != 0.0f) + (v.w != 0.0f);
        }
    } else {
        for (int k = lane; k < EE; k += 32) c += a[k] != 0.0f;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if (lane == 0) counts[g] = c;
}

// single block: every thread owns a contiguous run, block-level scan of the run totals in shared memory
__global__ void __launch_bounds__(1024) lsm_edge_scan_kernel(const int32_t* __restrict__ counts, long long* __restrict__ offsets,
                                                             long long num_graphs) {
    __shared__ long long part[1024];
    const int t = threadIdx.x, T = blockDim.x;
    const long long per = (num_graphs + T - 1) / T;
    const long long lo = (long long)t * per, hi = (lo + per) < num_graphs ? (lo + per) : num_graphs;
    long long s = 0;
    for (long long k = lo; k < hi; ++k) s += counts[k];
    part[t] = s;
    __syncthreads();
    for (int o = 1; o < T; o <<= 1) {       // Hillis-Steele inclusive scan over the T run totals
        const long long v = (t >= o) ? part[t - o] : 0;
        __syncthreads();
        part[t] += v;
        __syncthreads();
    }
    long long run = part[t] - s;            // exclusive prefix of this thread's run
    for (long long k = lo; k < hi; ++k) { offsets[k] = run; run += counts[k]; }
    if (t == T - 1) offsets[num_graphs] = part[T - 1];
}

__global__ void __launch_bounds__(256) lsm_edge_fill_kernel(const float* __restrict__ adj, const long long* __restrict__ offsets,
                                                            long long* __restrict__ edge_index, float* __restrict__ edge_attr,
                                                            long long num_graphs, int E, long long capacity) {
    const long long g = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (g >= num_graphs) return;
    const int lane = threadIdx.x & 31;
    const int EE = E * E;
    const float* a = adj + g * EE;
    long long pos = offsets[g];
    const long long node0 = g * E;
    long long* src = edge_index;
    long long* dst = edge_index + capacity;
    for (int k0 = 0; k0 < EE; k0 += 32) {
        const int k = k0 + lane;
        const float v = k < EE ? a[k] : 0.0f;
        const bool nz = v != 0.0f;
        const unsigned m = __ballot_sync(0xffffffffu, nz);
        if (nz) {
            const long long p = pos + __popc(m & ((1u << lane) - 1u));
            if (p < capacity) {
                const int row = k / E, col = k - row * E;
                src[p] = node0 + row; dst[p] = node0 + col; edge_attr[p] = v;
            }
        }
        pos += __popc(m);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Fused edge output (lsm_set_edge_output): the emit kernel itself writes the COO list, so the dense adjacency need not
// exist. It needs to know where each graph's edges start BEFORE it writes the first one; this kernel provides that.
//
//   lsm_edge_count_kernel<DYN,N,L>   one WARP per environment, reading the per-env emit record the agent kernel left:
//       the same exact float64 radius test and the same disconnected-entity masks as the emit kernel ->
//       counts[graph] for the N observer graphs of the env. The LAST block to finish (ticket counter) turns the counts of
//       this launch's env range into an exclusive prefix (edge_local) and the range total - no spinning, no second launch.
//   The emit kernel adds the totals of the earlier env ranges of the step (chunked launches: ordered by stream events).
// ---------------------------------------------------------------------------------------------------------------------
constexpr int kEdgeCountWarps = 4;
constexpr int kEdgeMaxEnvsPerBlock = 32;     // <= 32 envs x 32 agents = 1 024 graph counts per block in shared memory

// block-wide exclusive scan of one value per thread (T = 32 * kEdgeCountWarps threads); returns the exclusive prefix,
// *total = sum over the block. `s_w` is scratch of kEdgeCountWarps + 1 entries.
__device__ __forceinline__ long long edge_block_exscan(long long v, long long* s_w, long long* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const long long t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
    __syncthreads();                       // s_w may still be read from the previous call
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    long long base = 0, sum = 0;
#pragma unroll
    for (int w = 0; w < kEdgeCountWarps; ++w) { if (w < warp) base += s_w[w]; sum += s_w[w]; }
    *total = sum;
    return base + incl - v;
}

template <int DYN, int N, int L, int O>
__global__ void __launch_bounds__(32 * kEdgeCountWarps) lsm_edge_count_kernel(const __grid_constant__ KParams kp) {
    using REC = EmitRec<DYN, N, L, O>;
    constexpr int E = REC::E, W = REC::W;
    constexpr int T = 32 * kEdgeCountWarps;
    static_assert(sizeof(unsigned) * kEdgeCountWarps * (E * W + N * W) + sizeof(int) * kEdgeMaxEnvsPerBlock * N <= 40 * 1024,
                  "static shared memory of the edge-count kernel stays under the 48 KB static limit");
    __shared__ unsigned s_rowmask[kEdgeCountWarps][E * W];
    __shared__ unsigned s_keep[kEdgeCountWarps][N * W];
    __shared__ int s_cnt[kEdgeMaxEnvsPerBlock * N];
    __shared__ long long s_w[kEdgeCountWarps + 1];
    __shared__ bool s_last;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double r2_lt = kp.r2_lt, r2_nz = kp.r2_nz;
    pdl_launch_dependents();
    pdl_wait();
    // this block's CONTIGUOUS run of environments (so that its graph counts are one contiguous run of the prefix)
    const int c = kp.edge_envs_per_block;
    const int e0 = kp.env_begin + blockIdx.x * c;
    const int e1 = (e0 + c) < kp.env_end ? (e0 + c) : kp.env_end;
    // Every environment is counted from its emit record, also the ones a masked reset leaves alone: the emit kernel
    // re-emits those from the same (unchanged) record, while counts stored by an earlier launch may not describe it
    // (fresh buffers after lsm_set_edge_output are zero-filled).
    for (int ee = e0 + warp; ee < e1; ee += kEdgeCountWarps) {
        const REC& R = *reinterpret_cast<const REC*>(kp.emit_rec + (size_t)ee * sizeof(REC));
        unsigned* rowmask = s_rowmask[warp];
        unsigned* keep = s_keep[warp];
        // keep masks of the N observers (same expression as the emit kernel)
        unsigned dpre[W], dpost[W];
#pragma unroll
        for (int w = 0; w < W; ++w) {
            const int e = w * 32 + lane;
            bool pre = false, post = false;
            if (e < N) { pre = R.done[0][e] != 0; post = R.done[1][e] != 0; }
            else if (e < N + REC::M) {      // obstacles are never disconnected
                const int m = e - N, order = m / N, owner = m - order * N;
                pre = R.reached[0][owner] > order; post = R.reached[1][owner] > order;
            }
            dpre[w] = __ballot_sync(0xffffffffu, pre); dpost[w] = __ballot_sync(0xffffffffu, post);
        }
        for (int k = lane; k < N * W; k += 32) {
            const int w = k % W;
            const unsigned sel = kp.sel_tab[k];
            unsigned pr = 0u, po = 0u;
#pragma unroll
            for (int q = 0; q < W; ++q) if (q == w) { pr = dpre[q]; po = dpost[q]; }
            keep[k] = ~((po & sel) | (pr & ~sel));
        }
        // non-zero pattern of the thresholded distance matrix: d2 in float64 against the exact squared radius, and above
        // the largest d2 whose float32 distance is 0 (the emit kernel's test)
        double2 pb[W];
#pragma unroll
        for (int w = 0; w < W; ++w) pb[w] = (w * 32 + lane) < E ? R.pos[w * 32 + lane] : make_double2(0.0, 0.0);
        for (int a = 0; a < E; ++a) {
            const double2 pa = R.pos[a];
#pragma unroll
            for (int w = 0; w < W; ++w) {
                const double dx = pa.x - pb[w].x, dy = pa.y - pb[w].y;
                const double d2 = dx * dx + dy * dy;
                const unsigned m = __ballot_sync(0xffffffffu, (w * 32 + lane) < E && d2 < r2_lt && d2 > r2_nz);
                if (lane == 0) rowmask[a * W + w] = m;
            }
        }
        __syncwarp();
        // no connectivity flag changed in this step: every observer sees the same graph, count it once
        bool uniform = true;
#pragma unroll
        for (int w = 0; w < W; ++w) uniform = uniform && dpre[w] == dpost[w];
        for (int i = 0; i < (uniform ? 1 : N); ++i) {
            int cn = 0;
            for (int a = lane; a < E; a += 32) {
                if ((keep[i * W + (a >> 5)] >> (a & 31)) & 1u) {
#pragma unroll
                    for (int w = 0; w < W; ++w) cn += __popc(rowmask[a * W + w] & keep[i * W + w]);
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) cn += __shfl_xor_sync(0xffffffffu, cn, o);
            if (uniform) {
                for (int q = lane; q < N; q += 32) { kp.edge_counts[(size_t)ee * N + q] = cn; s_cnt[(ee - e0) * N + q] = cn; }
            } else if (lane == 0) { kp.edge_counts[(size_t)ee * N + i] = cn; s_cnt[(ee - e0) * N + i] = cn; }
        }
        __syncwarp();
    }
    __syncthreads();
    // exclusive prefix inside the block's run (each thread takes a few consecutive counts), block total
    {
        const int m = (e1 > e0 ? (e1 - e0) : 0) * N;
        const int per = (m + T - 1) / T;
        const int lo = tid * per, hi = (lo + per) < m ? (lo + per) : m;
        long long sum = 0;
        for (int k = lo; k < hi; ++k) sum += s_cnt[k];
        long long total;
        long long run = edge_block_exscan(sum, s_w, &total);
        for (int k = lo; k < hi; ++k) { kp.edge_local[(size_t)e0 * N + k] = (int)run; run += s_cnt[k]; }
        if (tid == 0) kp.edge_block_totals[kp.edge_block_ofs + blockIdx.x] = total;
    }
    // last block of this launch: prefix over the block totals -> base of every block, total of the range
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        const unsigned t = atomicAdd(kp.edge_tickets + kp.edge_range, 1u);
        s_last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    {
        const volatile long long* tot = kp.edge_block_totals + kp.edge_block_ofs;
        long long* base = kp.edge_block_base + kp.edge_block_ofs;
        const int G = (int)gridDim.x;
        long long running = 0;
        for (int t0 = 0; t0 < G; t0 += 8 * T) {
            long long v[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) { const int k = t0 + j * T + tid; v[j] = k < G ? tot[k] : 0; }   // all loads in flight
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                long long total;
                const long long ex = edge_block_exscan(v[j], s_w, &total);
                const int k = t0 + j * T + tid;
                if (k < G) base[k] = running + ex;
                running += total;
            }
        }
        if (tid == 0) { kp.edge_range_totals[kp.edge_range] = running; kp.edge_tickets[kp.edge_range] = 0u; }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// World graph of the renderer (SURVEY 8a row a16): `SafeAamScenario.update_graph` (navigation_graph_safe.py:996-1015),
// called at the top of every env.step (environment.py:964-965) on the distance matrix the previous step left behind -
// i.e. after graph_observation zeroed, IN PLACE, the rows / columns of every disconnected entity (:974-992, quirk Q1):
//     connect = (dists <= max_edge_dist) & (dists > 0)  ->  scipy COO (row-major)  ->  world.edge_list (2, nnz),
//     world.edge_weight = dists[row, col] (float64)
// ONE graph per environment, radius test INCLUSIVE (quirk Q7; the policy-facing adjacency is strict). Computed from the
// bound state: one warp per environment, pass 0 counts, pass 1 fills (offsets from lsm_edge_scan_kernel in between).
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) lsm_world_graph_kernel(const __grid_constant__ KParams kp, int pass, int32_t* __restrict__ counts,
                                                             const long long* __restrict__ offsets, long long* __restrict__ edge_index,
                                                             double* __restrict__ edge_weight, long long capacity) {
    const long long n = kp.b.num_envs;
    const long long env = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (env >= n) return;
    const int lane = threadIdx.x & 31;
    const int N = kp.N, M = kp.M, E = kp.E;
    const size_t fs = (size_t)n * N, ls = (size_t)n * M;
    auto pos = [&](int e, double& x, double& y, bool& disc) {
        if (e < N) {
            x = kp.b.agent_f64[LSM_AF_X * fs + env * N + e]; y = kp.b.agent_f64[LSM_AF_Y * fs + env * N + e];
            disc = kp.b.agent_i32[LSM_AI_DONE * fs + env * N + e] != 0;
        } else if (e < N + M) {
            const int m = e - N, order = m / N, owner = m - order * N;
            x = kp.b.landmarks[LSM_LF_X * ls + env * M + m]; y = kp.b.landmarks[LSM_LF_Y * ls + env * M + m];
            disc = kp.b.agent_i32[LSM_AI_REACHED * fs + env * N + owner] > order;
        } else {   // obstacle (extension): never disconnected
            const int k = e - N - M;
            x = kp.b.obstacles[((size_t)0 * n + env) * kp.O + k]; y = kp.b.obstacles[((size_t)1 * n + env) * kp.O + k];
            disc = false;
        }
    };
    long long p = pass ? offsets[env] : 0;
    int total = 0;
    for (int a = 0; a < E; ++a) {
        double ax, ay; bool adisc;
        pos(a, ax, ay, adisc);
        for (int b0 = 0; b0 < E; b0 += 32) {
            const int b = b0 + lane;
            bool on = false; double d2 = 0.0;
            if (b < E && !adisc) {
                double bx, by; bool bdisc;
                pos(b, bx, by, bdisc);
                const double dx = ax - bx, dy = ay - by;
                d2 = dx * dx + dy * dy;
                on = !bdisc && d2 < kp.r2_gt && d2 > 0.0;        // d <= R  <=>  d2 < min{t : sqrt(t) > R}
            }
            const unsigned m = __ballot_sync(0xffffffffu, on);
            if (pass && on) {
                const long long q = p + __popc(m & ((1u << lane) - 1u));
                if (q < capacity) { edge_index[q] = a; edge_index[capacity + q] = b; edge_weight[q] = sqrt(d2); }
            }
            p += __popc(m); total += __popc(m);
        }
    }
    if (!pass && lane == 0) counts[env] = total;
}

}  // namespace lsm

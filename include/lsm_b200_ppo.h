/*
 * lsm_b200_ppo.h - C ABI of the PPO-input kernels (liblsm_b200_ppo.so): the learner-side arithmetic that turns a
 * filled rollout buffer into PPO targets. Nothing here needs an environment handle, so these kernels live in their own
 * library, next to the simulator's liblsm_b200.so.
 *
 * Plain pointers and sizes only. Every array pointer is a DEVICE pointer owned by the caller. All launches go to the
 * cudaStream_t passed as `stream` (void*; NULL = default), on the caller's current device. No entry point synchronises.
 * Every function that can fail returns 0 on success, a non-zero code otherwise, and then lsm_ppo_last_error()
 * describes the failure (thread-local string): 2 = invalid arguments, 100 + cudaError_t = a launch failed.
 *
 * What each entry point replaces in the reference (paths relative to the reference root):
 *   lsm_compute_returns  GraphReplayBuffer.compute_returns (GAE / discounted, use_proper_time_limits, value normaliser)
 *                                                          onpolicy/utils/graph_buffer.py:285-373
 *                        + the advantage moments of GR_MAPPO.train (np.nanmean / np.nanstd over active entries)
 */
#ifndef LSM_B200_PPO_H
#define LSM_B200_PPO_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LSM_PPO_ABI_VERSION 1

int lsm_ppo_abi_version(void);
const char *lsm_ppo_last_error(void);

/* lsm_compute_returns: the returns recursion of DeviceGraphRolloutBuffer.compute_returns over C = columns independent
 * columns (C = n_rollout_threads * num_agents) and T steps, bit for bit what the torch loop computes: every operation is
 * one float32 operation rounded once, in the loop's order. Arrays are row-major [rows][C] float32.
 *
 *   d(v)            = v * value_scale + value_shift when both are given (ValueNorm / PopArt denormalize with
 *                     value_scale = sqrt(var), value_shift = mean, read on the device), else v
 *   use_gae         value_preds[T] = next_value;  gae = 0;  for t = T-1 .. 0:
 *                       delta = rewards[t] + gamma * d(value_preds[t+1]) * masks[t+1] - d(value_preds[t])
 *                       gae   = delta + gamma_lambda * masks[t+1] * gae
 *                       gae   = gae * bad_masks[t+1]                                  (use_proper_time_limits)
 *                       returns[t] = gae + d(value_preds[t])
 *                   returns[T] is left untouched.
 *   otherwise       returns[T] = next_value;  for t = T-1 .. 0:
 *                       r = returns[t+1] * gamma * masks[t+1] + rewards[t]
 *                       r = r * bad_masks[t+1] + (1 - bad_masks[t+1]) * d(value_preds[t])   (use_proper_time_limits)
 *                       returns[t] = r
 *
 * gamma and gamma_lambda are the float32 multipliers the torch loop applies: float32(gamma) and
 * float32(gamma * gae_lambda) with the product taken in double.
 *
 * Optional outputs of the same pass:
 *   advantages      [T][C]: returns[t] - d(value_preds[t])
 *   stats / stats64 the moments of those advantages over the entries with active_masks[t] != 0 (t < T), accumulated in
 *                   float64 and reduced in a fixed order (bitwise reproducible on one device): stats64 = {count, mean,
 *                   population std}, stats = {mean, std} rounded to float32. NaN mean and std when no entry is active,
 *                   as np.nanmean / np.nanstd give. They need active_masks and `scratch` (lsm_returns_scratch_bytes).
 */
typedef struct lsm_returns_io {
    int64_t T;                      /* steps, >= 0 */
    int64_t columns;                /* C >= 0 */
    const float *rewards;           /* [T][C] */
    float *value_preds;             /* [T+1][C]; row T is written in GAE mode */
    const float *next_value;        /* [C]; may alias row T of value_preds (GAE) or returns (discounted) */
    const float *masks;             /* [T+1][C] */
    const float *bad_masks;         /* [T+1][C]; read only with use_proper_time_limits (NULL allowed otherwise) */
    float *returns;                 /* [T+1][C] out */
    float *advantages;              /* [T][C] out, or NULL */
    const float *active_masks;      /* [T+1][C], needed with stats */
    const float *value_scale;       /* [1], or NULL (no denormalisation; then value_shift must be NULL too) */
    const float *value_shift;       /* [1], or NULL */
    void *scratch;                  /* lsm_returns_scratch_bytes(columns) bytes, 8-byte aligned, needed with stats */
    double *stats64;                /* [3] out: count, mean, std, or NULL */
    float *stats;                   /* [2] out: mean, std, or NULL (no moments when both stats and stats64 are NULL) */
    float gamma;
    float gamma_lambda;
    int32_t use_gae;
    int32_t use_proper_time_limits;
} lsm_returns_io;

int lsm_compute_returns(const lsm_returns_io *io, void *stream);

/* Bytes of the `scratch` lsm_compute_returns needs for the moments of `columns` columns (per-block partial moments). */
int64_t lsm_returns_scratch_bytes(int64_t columns);

#ifdef __cplusplus
}
#endif
#endif

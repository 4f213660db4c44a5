/* odg_mppi.h — sampling-MPC (MPPI) on the fused step kernel: BASELINE.json configs[4] "1024 action-sequence samples
 * x horizon 64 rolled out from a shared robot state, cost reduction on-device". The reference has no MPC code
 * (SURVEY §8d config 5): this is a new capability on the same hot path, expressed through the same env semantics —
 * a sample's cost is minus the sum of the walk-environment rewards (WalkEnvironment.py:81-109; the caller passes
 * OdgInfoPtrs.reward_unclipped, i.e. before the max(0, .) clip) along its rollout,
 * plus a penalty when it terminates (is_healthy, reward_calc:117-135).
 *
 * Per planning call: the caller broadcasts one robot state to N = num_samples environments of an OdgSim
 * (odg_set_state / odg_set_env_state), then for t in [0, T): odg_mppi_sample -> odg_step -> odg_mppi_accumulate,
 * and finally odg_mppi_reduce. Same conventions as odg.h.
 */
#ifndef ODG_MPPI_H
#define ODG_MPPI_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* action[n][a] = clamp(mean[a] + sigma * eps, -1, 1), eps ~ N(0,1) from Philox4x32-10 keyed by
 * (seed, n, iteration, t, block). mean_dev [A]; action_dev [N][A] (one row block of the [T][N][A] action tensor). */
int odg_mppi_sample(const float* mean_dev, float sigma, int n_samples, int act_dim, uint64_t seed, uint32_t iteration,
                    uint32_t t, float* action_dev, void* stream);

/* cost[n] += alive[n] ? -reward[n] : 0;  a sample that terminates pays `termination_cost` once and stops
 * accumulating (alive[n] = 0). cost_dev [N] f32, alive_dev [N] u8. */
int odg_mppi_accumulate(const float* reward_dev, const uint8_t* terminated_dev, int n_samples, float termination_cost,
                        float* cost_dev, uint8_t* alive_dev, void* stream);

/* The whole rollout of a plan in ONE launch (what opendog_b200.mppi.MPPI runs): for every sample n of `sim`
 * (created with auto_reset = 0; the caller has broadcast the shared start state with odg_set_state / odg_set_env_state)
 * and t in [0, horizon): draw action[t][n][:] exactly as odg_mppi_sample does, take the fused environment step of
 * odg_step, and accumulate cost[n] as odg_mppi_accumulate does (a terminated sample pays `termination_cost` once, stops
 * stepping and only keeps drawing its action rows). State stays on the SM between the steps of a sample's horizon; no
 * launch or grid-wide barrier separates them. mean_dev [T][A]; actions_dev [T][N][A]; cost_dev [N] (overwritten).
 * `iteration_dev` (nullable) points to a device-side plan counter that overrides `iteration`: a CUDA graph that
 * increments it replays with fresh noise every plan. */
struct OdgSim;
int odg_mppi_rollout(struct OdgSim* sim, const float* mean_dev, float sigma, int horizon, uint64_t seed, uint32_t iteration,
                     const uint32_t* iteration_dev, float termination_cost, float* actions_dev, float* cost_dev, void* stream);

/* Information-theoretic MPPI update, one block, fixed summation order (deterministic):
 *   w[n] = exp(-(cost[n] - min cost) / lambda);  mean_out[t][a] = sum_n w[n] action[t][n][a] / sum_n w[n]
 * actions_dev [T][N][A]; mean_out_dev [T][A]; stats_dev [4] f32 = (min cost, mean cost, sum w, argmin) nullable.
 * Non-finite costs (a sample whose rollout state went NaN or infinite): only samples with a finite cost take part in
 * the min, the argmin, the mean cost and the weights; a non-finite cost gets weight exactly 0, so the result is that of
 * the same costs with it replaced by any finite value whose weight underflows to 0. If no cost is finite, mean_out = 0
 * and stats = (+inf, NaN, 0, -1). With every cost finite the arithmetic is the plain formula above.
 * (tests/test_gpu_mppi_numerics.py) */
int odg_mppi_reduce(const float* cost_dev, const float* actions_dev, int horizon, int n_samples, int act_dim,
                    float lambda, float* mean_out_dev, float* stats_dev, void* stream);

/* ---- Batched MPPI: G robots planned in one launch each, each from its own start state (opendog_b200.mppi.BatchedMPPI).
 * A samples handle of N = G * S environments holds G groups of S samples; sample n = g * S + s belongs to group g.
 * Per plan: odg_mppi_broadcast -> odg_mppi_rollout_groups -> odg_mppi_reduce_groups, no host round trip.
 *
 * Copy robot `first_robot + g` of `robots` into samples [g S, (g + 1) S) for g in [0, groups), S = samples.n / groups,
 * in one launch on the device (SoA to SoA): qpos, qvel, the solver's qacc warm start, step counter, gait index, gait
 * matches, last action, desired velocity and `fresh` — every per-environment field the env-step reads. Invariant: when
 * the two handles share model and config, a sample stepped with its robot's action reproduces that robot's step bit
 * for bit (which is why the warm start is copied, not zeroed). ODG_ERR_INVALID, before any device work, for null
 * handles, handles on different devices, different nq / nv / nu / task, groups < 1, first_robot < 0,
 * first_robot + groups > robots.n, samples.n % groups != 0, or a samples handle created with auto_reset = 1. */
int odg_mppi_broadcast(struct OdgSim* samples, const struct OdgSim* robots, int first_robot, int groups, void* stream);

/* odg_mppi_rollout for `groups` groups of S = sim.n / groups samples: sample n = g * S + s follows the nominal
 * sequence mean[g] and draws its noise exactly as a single-robot plan draws it for sample s with the 64-bit key
 * seed + g. So group g equals odg_mppi_rollout(seed + g) on an S-sample handle holding the same start state (e.g.
 * filled by odg_mppi_broadcast(first_robot = g, groups = 1)), bit for bit, action rows and costs; odg_mppi_rollout is
 * the groups = 1 case. mean_dev [G][T][A]; actions_dev [T][N][A]; cost_dev [N]. ODG_ERR_INVALID when groups < 1 or
 * sim.n % groups != 0, and for the arguments odg_mppi_rollout refuses. */
int odg_mppi_rollout_groups(struct OdgSim* sim, int groups, const float* mean_dev, float sigma, int horizon, uint64_t seed,
                            uint32_t iteration, const uint32_t* iteration_dev, float termination_cost, float* actions_dev,
                            float* cost_dev, void* stream);

/* odg_mppi_reduce per group: one 1024-thread block per group, the same fixed tree and in-order sample sums, so group g
 * equals odg_mppi_reduce on a contiguous copy of actions[:, g S:(g + 1) S] bit for bit; odg_mppi_reduce is the
 * groups = 1 case. actions_dev [T][G S][A]; cost_dev [G S]; mean_out_dev [G][T][A]; stats_dev [G][4] nullable, with
 * stats[g][3] the argmin within group g. samples_per_group <= 12000. Non-finite costs as in odg_mppi_reduce, per group:
 * a group with no finite cost writes mean_out[g] = 0 (the nominal an ended episode restarts from) and
 * stats[g] = (+inf, NaN, 0, -1); the other groups are unaffected. */
int odg_mppi_reduce_groups(const float* cost_dev, const float* actions_dev, int horizon, int groups, int samples_per_group,
                           int act_dim, float lambda, float* mean_out_dev, float* stats_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ODG_MPPI_H */

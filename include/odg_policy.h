/* odg_policy.h — C ABI of the rollout side of libodgsim: the policy MLP forward on tensor cores, GAE and
 * advantage statistics. Companion of odg.h (same conventions: plain pointers and sizes, caller-owned device
 * buffers, `stream` = cudaStream_t as void*, 0 / negative OdgStatus, never throws).
 *
 * Reference interfaces replaced (paths relative to /root/reference/Code/mujoco):
 *   ActorCritic.forward + dist.sample() + log_prob().sum(-1)      sim2real/train.py:132-149, 540-545
 *   the GAE loop and advantage normalisation                      sim2real/train.py:557-564
 * The reference runs the network with batch size 1 and a host<->device round trip per environment step; here one
 * launch serves the whole batch of environments and nothing leaves HBM.
 */
#ifndef ODG_POLICY_H
#define ODG_POLICY_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct OdgPolicy OdgPolicy;

#define ODG_POLICY_H1 512      /* nn.Linear(state_dim, 512)   sim2real/train.py:136,141 */
#define ODG_POLICY_H2 256      /* nn.Linear(512, 256)         sim2real/train.py:137,142 */
#define ODG_POLICY_MAX_STATE 64
#define ODG_POLICY_MAX_ACTION 16

/* Weights of one ActorCritic in the layout of its torch state_dict (float32, device pointers):
 * actor.{0,2,4}.weight [out][in] row-major, actor.{0,2,4}.bias [out], critic.{0,2,4}.*, action_log_std [A].
 * Shapes follow the handle's hidden widths h1 / h2: weight 0 [h1][S], weight 2 [h2][h1], weight 4 [A or 1][h2]. */
typedef struct OdgPolicyWeights {
  const float* actor_w[3];
  const float* actor_b[3];
  const float* critic_w[3];
  const float* critic_b[3];
  const float* action_log_std;
} OdgPolicyWeights;

/* Replaces `ActorCritic(state_dim, action_dim, std).to(device)` (sim2real/train.py:533). state_dim <= 64,
 * action_dim <= 16; hidden sizes are the reference's 512 / 256. */
int odg_policy_create(int state_dim, int action_dim, int device, OdgPolicy** out);
/* The same with the hidden widths given: (h1, h2) = (512, 256) is odg_policy_create; (1024, 512) is the terrain trainer's
 * ActorCritic (sim2real/train2.py:149-157, 12 -> 1024 -> 512 -> 8). Any other widths, or state_dim / action_dim out of
 * range, return ODG_ERR_INVALID before the device is looked at. The 1024 / 512 forward has the same contract as the 512 / 256
 * one (bf16 operands, fp32 accumulation, the same noise for the same key); its output layer is computed on CUDA cores from
 * the bf16 hidden-2 values and bf16 weights with fp32 sums. odg_policy_load and odg_policy_forward serve both. */
int odg_policy_create_hidden(int state_dim, int action_dim, int h1, int h2, int device, OdgPolicy** out);
void odg_policy_destroy(OdgPolicy* p);

/* Replaces `agent.load_state_dict(...)` / the optimiser's in-place update: converts the fp32 weights to the
 * bf16 tensor-core operand layout kept by the handle. Call after every optimiser step. */
int odg_policy_load(OdgPolicy* p, const OdgPolicyWeights* w, void* stream);

/* Replaces `dist, value = agent(state); action = dist.sample(); logp = dist.log_prob(action).sum(-1)`
 * (sim2real/train.py:542-543) for n rows at once.
 *   obs_dev    [n][state_dim] f32
 *   mean_dev   [n][action_dim] f32   tanh output of the actor (dist.mean; the export path uses it, :613)
 *   value_dev  [n] f32               critic output
 *   action_dev [n][action_dim] f32   mean + exp(log_std) * eps, eps ~ N(0,1) from Philox4x32-10 keyed by
 *                                    (seed, first_row_id + row, step + *step_base_dev); NULL = no sampling.
 *                                    step_base_dev (nullable, u32 in device memory) lets a captured CUDA graph
 *                                    advance the noise stream between replays
 *   logp_dev   [n] f32               sum over action dims of the Normal log-density of the sampled action; NULL ok
 * bf16 operands, fp32 accumulation (tcgen05.mma, accumulators in TMEM). */
int odg_policy_forward(OdgPolicy* p, const float* obs_dev, int n, float* mean_dev, float* value_dev,
                       float* action_dev, float* logp_dev, uint64_t seed, uint32_t step,
                       const uint32_t* step_base_dev, int first_row_id, void* stream);

/* Replaces the GAE loop (sim2real/train.py:557-561), batched over n environments and T steps:
 *   delta = r[t] + gamma * V[t+1] * (1 - done[t]) - V[t];  A[t] = delta + gamma*lambda*(1 - done[t]) * A[t+1]
 *   reward_dev [T][n], value_dev [T+1][n] (value_dev[T] = bootstrap value), done_dev [T][n] u8
 *   adv_dev, ret_dev [T][n] (returns = adv + value)
 *   stats_dev [3] f64: sum(adv), sum(adv^2), count — summed in a fixed order (deterministic); all-reduce these
 *   across ranks (NCCL) before odg_normalize_advantages when environments are sharded over GPUs. */
int odg_gae(const float* reward_dev, const float* value_dev, const uint8_t* done_dev, int T, int n, float gamma,
            float lambda, float* adv_dev, float* ret_dev, double* stats_dev, void* stream);

/* Replaces `(adv - adv.mean()) / (adv.std() + 1e-8)` (sim2real/train.py:564; torch.std is the unbiased one)
 * using the (possibly all-reduced) statistics. */
int odg_normalize_advantages(float* adv_dev, long long count, const double* stats_dev, void* stream);

/* PPO update phase (sim2real/train.py:566-585: `loss.backward()` through `nn.Tanh` + `nn.Linear` of the hidden layers):
 * grad_x = grad_y * (1 - y*y) for a [rows][cols] bf16 activation gradient (torch's tanh_backward) AND, in the same pass
 * over the data, bias_grad[cols] (f32) = the column sums of grad_x = the bias gradient of the Linear that produced the
 * tanh's input. Deterministic (fixed summation order). cols = 8 x a power of two, <= 2048; grad_y, y and grad_x 16-byte
 * aligned (ODG_ERR_INVALID otherwise); grad_x must not overlap the inputs.
 * scratch_dev: odg_tanh_backward_bias_scratch_floats(cols) floats of device memory, owned by the caller (so that the call
 * can be captured in a CUDA graph). */
int odg_tanh_backward_bias_scratch_floats(int cols);
int odg_tanh_backward_bias(const void* grad_y_bf16, const void* y_bf16, void* grad_x_bf16, float* bias_grad_dev,
                           float* scratch_dev, long long rows, int cols, void* stream);

/* PPO update phase: the clipped-surrogate loss of one minibatch (stable-baselines3's PPO objective with the
 * hyper-parameters of train/train.py:117-130; the update of sim2real/train.py:566-569, actor_loss = -(logp*adv).mean(), is
 * its special case clip = +inf with logp_old = logp) and its gradients in one pass over the samples. Inputs f32: mean [B][A] (the actor's output),
 * value [B], log_std [A], action [B][A], logp_old / adv / ret [B]. Outputs: loss_dev [1] = pg + vf_coef*vf - ent_coef*ent,
 * terms_dev [4] = {loss, pg, vf, entropy} with pg = mean(-min(r*adv, clamp(r, 1-clip, 1+clip)*adv)), r = exp(logp - logp_old),
 * vf = mean((value - ret)^2), entropy = sum_k(0.5 + 0.5 log 2pi + log_std[k]); grad_mean_dev [B][A], grad_value_dev [B],
 * grad_log_std_dev [A] = d loss / d (those inputs), with torch.min's / torch.clamp's gradient conventions (ties split
 * evenly, clamp ends pass). Deterministic. 1 <= A <= 16. scratch_dev: odg_ppo_loss_scratch_floats() floats, caller-owned. */
int odg_ppo_loss_scratch_floats(void);
int odg_ppo_loss(const float* mean_dev, const float* value_dev, const float* log_std_dev, const float* action_dev,
                 const float* logp_old_dev, const float* adv_dev, const float* ret_dev, long long B, int A, float clip,
                 float vf_coef, float ent_coef, float* loss_dev, float* terms_dev, float* grad_mean_dev,
                 float* grad_value_dev, float* grad_log_std_dev, float* scratch_dev, void* stream);

/* PPO update phase, forward: y = tanh(x) for `count` bf16 values (a multiple of 8; x and y 16-byte aligned, ODG_ERR_INVALID otherwise; y may be x) with the
 * hardware tanh the rollout kernel's epilogue uses (odg_policy_forward), so that the update-time policy evaluates the same
 * function as the policy that produced logp_old. Replaces nn.Tanh of sim2real/train.py:136-147 on bf16 activations. */
int odg_tanh_bf16(const void* x_bf16, void* y_bf16, long long count, void* stream);

long long odg_policy_launch_count(const OdgPolicy* p);

#ifdef __cplusplus
}
#endif
#endif /* ODG_POLICY_H */

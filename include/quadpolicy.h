/*
 * quadpolicy.h -- C-ABI of the fused policy forward used by the device-resident rollouts (SURVEY.md 8 f1).
 *
 * Replaces, for rollout collection, the per-step forward of the reference's policy
 * (priban42/quad-swarm-rl-stable-baselines3, paths relative to the reference root):
 *
 *   qp_create / qp_destroy   ActorCriticPolicyCustomSeparateWeights.__init__ / _build   swarm_rl/models/ActorCriticPolicyCustom.py:284-411
 *                            QuadMultiEncoder.__init__ (one per tower)                  swarm_rl/models/quad_multi_model.py:250-331
 *   qp_set_weights           the state_dict of one tower (nn.Linear weights [out, in], biases)
 *   qp_gae                   stable_baselines3 RolloutBuffer.compute_returns_and_advantage as driven by PPO.collect_rollouts
 *                            (swarm_rl/sb_train.py:54-99 -> model.learn): one launch over the device-resident rollout
 *   qp_bias_tanh[_mean][_backward]   the elementwise half of the dense tanh layers under autograd in the PPO update (evaluate_actions)
 *   qp_forward               ActorCriticPolicyCustom.forward / predict_values: action mean of the actor tower and value of the
 *                            critic tower for a batch of observations           ActorCriticPolicyCustom.py:430-480,
 *                            QuadMultiEncoder.forward                           quad_multi_model.py:333-354,
 *                            QuadNeighborhoodEncoderDeepsets.forward            quad_multi_model.py:16-41
 *
 * Architecture built: self encoder S -> 256 -> 256, deep-sets neighbour encoder ('mean_embed') W -> 256 -> 256 averaged over V neighbours,
 * optional obstacle encoder O -> 256 -> 256, feed-forward [self | neighbour | obstacle] (512 or 768) -> 512, all tanh; heads 512 -> A (actor) and 512 -> 1 (critic).
 * bf16 operands, fp32 accumulation (tcgen05 tensor cores); biases, heads and outputs fp32.  Sampling and log-probabilities stay with the
 * caller (state-independent log-std diagonal Gaussian, ActorCriticPolicyCustom.py:312).  Not built: the 'attention' and 'mlp' neighbour
 * encoders, widths other than 256.
 *
 * All pointers are CUDA device addresses unless stated; `stream` is a cudaStream_t passed as void*.  Calls return 0 or a negative
 * qp_status; qp_last_error() gives a message.  A handle is bound to one device and is not thread-safe.
 */
#ifndef QUADPOLICY_H_
#define QUADPOLICY_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Version 2 appended obst_dim to qp_config and the obst_* fields to qp_tower_weights.  qp_create still accepts a version-1 config (the first six
 * fields): such a handle has no obstacle encoder and never reads the obst_* fields of qp_tower_weights. */
#define QP_API_VERSION 2

typedef enum { QP_OK = 0, QP_ERR_NULL = -1, QP_ERR_BAD_CONFIG = -2, QP_ERR_CUDA = -3 } qp_status;

typedef struct {
    int32_t api_version; /* QP_API_VERSION */
    int32_t self_dim;    /* S: 18 / 19 / 24 (quad_utils.py:30-38); S <= 24 */
    int32_t nbr_dim;     /* W: 6 for pos_vel (quad_utils.py:40-58); W <= 8 */
    int32_t num_nbr;     /* V: neighbour rows in the observation, 0 = no neighbour encoder */
    int32_t hidden;      /* rnn_size: 256 (the only width built) */
    int32_t act_dim;     /* A <= 8 */
    int32_t obst_dim;    /* O: obstacle observation columns (9 = the SDF patch), 0 = no obstacle encoder; O <= 24 (since version 2) */
} qp_config;

/* one tower's parameters: device pointers to fp32 arrays in nn.Linear layout (weight [out, in] row-major, bias [out]) */
typedef struct {
    const float *self_w1, *self_b1; /* [256, S], [256] */
    const float *self_w2, *self_b2; /* [256, 256], [256] */
    const float *nbr_w1, *nbr_b1;   /* [256, W], [256]   (ignored when num_nbr == 0) */
    const float *nbr_w2, *nbr_b2;   /* [256, 256], [256] */
    const float *ff_w, *ff_b;       /* [512, 512] ([512, 768] when obst_dim > 0), [512]; input = [self | neighbour | obstacle encoder];
                                       without neighbours (num_nbr == 0) the neighbour block must be zeros */
    const float *head_w, *head_b;   /* actor: [A, 512], [A]; critic: [1, 512], [1] */
    const float *obst_w1, *obst_b1; /* [256, O], [256]   (since version 2; read only when obst_dim > 0) */
    const float *obst_w2, *obst_b2; /* [256, 256], [256] */
} qp_tower_weights;

typedef struct qp_policy qp_policy;

size_t qp_config_size(void);
const char *qp_last_error(const qp_policy *p);
int qp_create(const qp_config *cfg, int device, qp_policy **out);
int qp_destroy(qp_policy *p);
int64_t qp_launch_count(const qp_policy *p);

/* (re)pack one tower's weights into the kernel's bf16 tile images; tower 0 = actor, 1 = critic.  Asynchronous on `stream`: the source arrays must
 * stay valid (and unchanged) until the stream has passed this call; a later qp_forward on the same stream sees the new weights. */
int qp_set_weights(qp_policy *p, int tower, const qp_tower_weights *w, void *stream);

/* obs: [n, obs_stride] fp32 (self block first, then V neighbour rows of W values, then the O obstacle columns, as Appendix B of SURVEY.md),
 * obs_stride >= S + V * W + O; mean: [n, A]; value: [n].  One kernel launch, nothing touches the host. */
int qp_forward(qp_policy *p, const float *obs, int n, int obs_stride, float *mean, float *value, void *stream);

/* GAE over a rollout held on the device: rewards / values [T, n] fp32, dones [T, n] bytes (dones[t] = the transition produced by step t
 * ended its episode), last_values [n] = V(s_T); writes advantages and returns [T, n].  One launch; no handle needed. */
int qp_gae(const float *rewards, const float *values, const uint8_t *dones, const float *last_values, int T, int n, float gamma, float lam,
           float *advantages, float *returns, void *stream);

/* The elementwise half of a dense tanh layer in the PPO update (ActorCriticPolicyCustom.evaluate_actions -> QuadMultiEncoder.forward under
 * autograd): y = tanh(z + bias) and, in one pass, its backward grad_z = grad_y * (1 - y^2) with grad_bias = column sums of grad_z.
 * z, y, grad_* are [n, h] row-major, bf16 (is_bf16 != 0, the autocast path) or fp32; bias / grad_bias are fp32 [h]; h even, <= 2048.
 * The [n, h] pointers must be aligned to one element pair (8 bytes fp32, 4 bytes bf16), else QP_ERR_BAD_CONFIG; with h % 8 == 0 and
 * 16-byte alignment the calls take the faster 8-column form. */
int qp_bias_tanh(const void *z, const float *bias, int n, int h, int is_bf16, void *y, void *stream);
int qp_bias_tanh_backward(const void *grad_y, const void *y, int n, int h, int is_bf16, void *grad_z, float *grad_bias, void *stream);

/* Backward of a FIRST tanh layer with at most 8 inputs (the deep-sets phi, 6 -> 256 over n * V rows) whose input needs no gradient: grad_bias [h] and
 * grad_weight [h, in_dim] (nn.Linear layout) from one pass over grad_y and y; grad_z is never written.  x: fp32 [n, in_dim] row-major; `workspace`:
 * device scratch of qp_bias_tanh_backward_first_workspace(h, in_dim) bytes (per-block partial sums, no atomics). */
size_t qp_bias_tanh_backward_first_workspace(int h, int in_dim);
int qp_bias_tanh_backward_first(const void *grad_y, const void *y, const float *x, int n, int h, int in_dim, int is_bf16, void *workspace,
                                float *grad_bias, float *grad_weight, void *stream);

/* Tail of the deep-sets neighbour encoder (QuadNeighborhoodEncoderDeepsets.forward, quad_multi_model.py:35-40): y = tanh(z + bias) on [n * V, h]
 * and mean [n, h] = the average of each group of V consecutive rows, in one pass; the backward takes grad_mean [n, h] and writes
 * grad_z [n * V, h] = grad_mean[group] / V * (1 - y^2) and grad_bias.  h a multiple of 8, pointers 16-byte aligned. */
int qp_bias_tanh_mean(const void *z, const float *bias, int n, int V, int h, int is_bf16, void *y, void *mean, void *stream);
int qp_bias_tanh_mean_backward(const void *grad_mean, const void *y, int n, int V, int h, int is_bf16, void *grad_z, float *grad_bias, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* QUADPOLICY_H_ */

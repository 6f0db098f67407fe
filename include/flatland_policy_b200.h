/* flatland_policy_b200.h — C ABI of the batched policy forward pass (SURVEY.md §8 f1): the consumer that
 * follows the step/observation path immediately, evaluated for all E*N agents of a lock-step batch from the
 * observation tensors where fl_observe left them (include/flatland_b200.h), without a host round trip.
 *
 * Replaces, in the reference (paths relative to the reference repository root):
 *   solution/nn/net_tree.py:73-98   Network.forward (attr MLP, 3 x MultiheadAttention block, actor / critic heads)
 *   solution/nn/TreeLSTM.py:34-154  TreeLSTM.forward / _run_lstm (child-sum style Tree-LSTM over the 31-node trees)
 *   solution/eval_env.py:76         forest[forest == inf] = -1
 *   solution/plfActor.py:15-44      Actor.get_actions / _choose_action (soft choice, generator re-seeded with 42)
 * The reference runs these through torch on the CPU with batch 1 (plfActor.py:18-20); there is no native
 * interface to bind, so the boundary is this C ABI under the Python class `BatchedActor`
 * (flatland-marl_b200/policy.py) that keeps `Actor.get_actions`' meaning.
 *
 * Arithmetic: bf16 operands, fp32 accumulation on the 5th-generation tensor cores (tcgen05.mma, accumulators in
 * TMEM); gates, GELU, softmax in fp32.  Tolerance against the fp32 reference is stated in tests/test_gpu_policy.py.
 *
 * Conventions as in flatland_b200.h: plain device pointers, `stream` is a cudaStream_t passed as void*, return
 * 0 or an FlStatus / CUDA error code, no allocation inside the library.
 */
#ifndef FLATLAND_POLICY_B200_H
#define FLATLAND_POLICY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FL_POLICY_ABI_VERSION 1
#define FL_POLICY_HIDDEN 128 /* NetworkConfig.hidden_sz = tree_embedding_sz (solution/impl_config.py:23-25) */
#define FL_POLICY_EMB 256
#define FL_POLICY_HEADS 4
#define FL_POLICY_LAYERS 3
#define FL_POLICY_MAX_LEVELS 11 /* node_order of a 31-node ternary tree is at most 10 */

/* Device-resident parameters.  Matrices are bf16 (raw uint16), row-major [out][in] exactly as nn.Linear stores
 * them, `in` zero-padded to the stated width; biases are fp32.  flatland-marl_b200/policy.py packs them from a
 * reference state_dict. */
typedef struct FlPolicyWeights {
    /* Tree-LSTM.  The gate biases ride in the matrix product: the node-feature operand carries a constant 1 in column 12
     * and column 12 of tree_wiou / column 140 of tree_ufwf holds the bias.  Rows of the sigmoid gates (i: 0..127, o:
     * 128..255 of tree_uiou / tree_wiou, and all of tree_ufwf) are stored multiplied by 1/2, because the kernels
     * evaluate sigmoid(2z) as 0.5 tanh(z) + 0.5 (one MUFU operation). */
    const uint16_t *tree_uiou;  /* [384][384]  tree_lstm.U_iou.weight (i, o rows x 1/2) */
    const uint16_t *tree_wiou;  /* [384][16]   tree_lstm.W_iou.weight | col 12: W_iou.bias (i, o rows x 1/2) */
    const uint16_t *tree_wc;    /* [128][384]  tree_lstm.W_c.weight */
    const uint16_t *tree_ufwf;  /* [128][144]  (tree_lstm.U_f.weight | tree_lstm.W_f.weight | col 140: W_f.bias) x 1/2 */
    const float *tree_b_iou;    /* [384] unscaled, kept for reference (not read by the kernels) */
    const float *tree_b_c;      /* [128] */
    const float *tree_b_f;      /* [128] unscaled, kept for reference (not read by the kernels) */
    const uint16_t *attr_w[4];  /* [256][128 (83 used)], [256][256], [256][256], [128][256]  attr_embedding.{0,2,4,6} */
    const float *attr_b[4];
    const uint16_t *tf_wqkv[FL_POLICY_LAYERS]; /* [768][256] transformer.l.attention.in_proj_weight */
    const float *tf_bqkv[FL_POLICY_LAYERS];
    const uint16_t *tf_wo[FL_POLICY_LAYERS];   /* [256][256] attention.out_proj.weight (kept for reference, not read: folded below) */
    const float *tf_bo[FL_POLICY_LAYERS];
    const uint16_t *tf_wm[FL_POLICY_LAYERS];   /* [256][512] att_mlp.0.weight with the out-projection folded in:
                                                  [W1 | W2 Wo], so that the layer reads cat(input, attention heads) */
    const float *tf_bm[FL_POLICY_LAYERS];      /* att_mlp.0.bias + W2 out_proj.bias */
    const uint16_t *head_w1;    /* [512][512] rows 0..255 actor_net.0.weight, rows 256..511 critic_net.0.weight */
    const float *head_b1;       /* [512] */
    const uint16_t *head_w2a;   /* [128][256] actor_net.2.weight */
    const uint16_t *head_w2c;   /* [128][256] critic_net.2.weight */
    const float *head_b2;       /* [256] actor_net.2.bias | critic_net.2.bias */
    const float *head_w3;       /* [6][128] fp32: rows 0..4 actor_net.4.weight, row 5 critic_net.4.weight */
    const float *head_b3;       /* [6] */
} FlPolicyWeights;

int fl_policy_abi_version(void);

/* Bytes of device scratch fl_policy_forward needs for n_agents_total = E*N agents (256-byte aligned blocks). */
size_t fl_policy_workspace_bytes(int64_t n_agents_total);

/* Network.forward for E environments of N agents each.  Inputs are the tensors fl_observe wrote
 * (d_agent_attr [E][N][83] f32, d_forest [E][N][31][12] f32 with +inf still in place, d_adjacency [E][N][30][3],
 * d_node_order [E][N][31], d_edge_order unused: edge order is node_order[parent]).
 * Outputs: d_logits [E][N][5] f32 (net_tree.py:94-96 worker_action), d_value [E] f32 (critic mean over agents,
 * net_tree.py:107-110).  d_workspace: fl_policy_workspace_bytes(E*N) bytes. */
int fl_policy_forward(const FlPolicyWeights *w, void *d_workspace, size_t workspace_bytes, int64_t E, int64_t N,
                      const float *d_agent_attr, const float *d_forest, const int32_t *d_adjacency,
                      const int32_t *d_node_order, float *d_logits, float *d_value, void *stream);

/* The same forward pass in the reference's own arithmetic: fp32 operands and accumulation on the CUDA cores, exact erf-GELU /
 * sigmoid / tanh, the reference's unfolded parameters (csrc/policy/policy_f32.cuh).  d_weights: FL_POLICY_F32_TENSORS device
 * pointers to the fp32 tensors of the reference state_dict in its registration order (solution/nn/net_tree.py:33-72,
 * TreeLSTM.py:12-32; flatland-marl_b200/policy_weights.py:weight_spec lists names and shapes).  Logits and values agree with
 * the reference network to summation-order rounding (tests: 1e-4 absolute); about ten times slower than the tensor-core
 * path.  It is the training forward of fl_policy_ppo_grad_f32 run on a smaller workspace that keeps no activations for a
 * backward pass.  Synchronises `stream` once (per-level node counts).  d_workspace: fl_policy_workspace_bytes_f32(E*N)
 * bytes (0 for n_agents_total <= 0).  FL_ERR_BAD_ARG before any CUDA call for a NULL pointer (also among d_weights), E or
 * N <= 0, E*N*31 >= 2^31 (node ids are 32-bit) or a workspace that is too small. */
#define FL_POLICY_F32_TENSORS 46
size_t fl_policy_workspace_bytes_f32(int64_t n_agents_total);
int fl_policy_forward_f32(const float *const *d_weights, void *d_workspace, size_t workspace_bytes, int64_t E, int64_t N,
                          const float *d_agent_attr, const float *d_forest, const int32_t *d_adjacency,
                          const int32_t *d_node_order, float *d_logits, float *d_value, void *stream);

/* PPO loss and gradients of the fp32 network (csrc/policy/policy_f32_grad.cuh): one training forward with the arithmetic of
 * fl_policy_forward_f32 (d_logits [E][N][5], d_value [E] bit-identical to it), the loss below, and its gradient with respect
 * to every parameter, in fp32 on the CUDA cores.
 *
 * Inputs as fl_policy_forward_f32, plus per agent d_valid_actions [E][N][5] u8, d_actions [E][N] u8 (the actions taken,
 * 0..4; a larger value is read as 4), d_old_log_probs [E][N] f32 (log pi_old, as fl_policy_sample_actions wrote it), and
 * per row d_advantages, d_returns [E] f32, d_acted [E] u8.  With log pi_new(a) = (x_a - max) - log(sum of expf(x_j - max)) over the valid actions
 * j in action order (the arithmetic of fl_policy_sample_actions), r = exp(log pi_new - log pi_old), A, R, V the row's
 * advantage, return and critic value (mean over agents):
 *   S      = the agents of rows with acted = 1 that have at least one valid action; rows = the rows with acted = 1
 *   L_pol  = mean_S( -min(r A, clip(r, 1 - clip_eps, 1 + clip_eps) A) ), the gradient flowing through r A where
 *            r A <= clip(r) A (ties included)
 *   H      = entropy of the masked softmax
 *   L      = L_pol - ent_coef mean_S(H) + vf_coef mean_rows((V - R)^2)
 * An empty set contributes 0.  Agents with no valid action have log-probability 0 and no gradient.
 * d_grads: FL_POLICY_F32_TENSORS device pointers, the shapes of d_weights (weight_spec order), overwritten with dL/dparameter.
 * d_stats [8] f32: L_pol, mean_rows((V - R)^2), mean_S(H), approximate KL mean_S(log pi_old - log pi_new), clip fraction
 * mean_S(|r - 1| > clip_eps), |S|, the number of acted rows, L.
 * Deterministic: no floating-point atomics; weight gradients reduce over fixed row chunks, then in chunk order.  Two calls
 * with the same inputs give the same bytes.  Synchronises `stream` once (per-level node counts), like the fp32 forward.
 * d_workspace: fl_policy_workspace_bytes_grad_f32(E*N) bytes (about 250 KB per agent).  FL_ERR_BAD_ARG before any CUDA call
 * for a NULL pointer (also among d_weights / d_grads), E or N <= 0, a workspace that is too small or clip_eps <= 0. */
typedef struct FlPpoParams {
    float clip_eps, vf_coef, ent_coef;
} FlPpoParams;
size_t fl_policy_workspace_bytes_grad_f32(int64_t n_agents_total);
int fl_policy_ppo_grad_f32(const float *const *d_weights, void *d_workspace, size_t workspace_bytes, int64_t E, int64_t N,
                           const float *d_agent_attr, const float *d_forest, const int32_t *d_adjacency,
                           const int32_t *d_node_order, const uint8_t *d_valid_actions,
                           const uint8_t *d_actions, const float *d_old_log_probs,
                           const float *d_advantages, const float *d_returns,
                           const uint8_t *d_acted,
                           const FlPpoParams *params,
                           float *const *d_grads,
                           float *d_logits, float *d_value, float *d_stats, void *stream);

/* The same loss, statistics and outputs through the same graph, with the dense products on the tensor cores
 * (csrc/policy/policy_bf16_grad.cuh).  Arguments, workspace, argument errors, determinism and the one host synchronisation
 * are those of fl_policy_ppo_grad_f32; the arithmetic differs in one place only:
 *   - The tensor-core layers: the weights U_iou, U_f, W_c (Tree-LSTM), attr_embedding.{0,2,4,6}, per transformer layer
 *     in_proj, out_proj and att_mlp.0, actor_net.{0,2} and critic_net.{0,2}.  For each of them the forward X W^T, the input
 *     gradient dY W and the weight gradient dY^T X run as tcgen05.mma kind::f16: both operands are the fp32 values rounded
 *     to bf16 (round to nearest even), the products accumulate in fp32.  The bias gradient is the fp32 sum over rows of the
 *     unrounded dY, over fixed row chunks and then in chunk order.
 *   - Everything else is the fp32 path's arithmetic in its kernels: the 12-feature node terms W_iou x, W_f x and their weight
 *     gradients, actor_net.4 and critic_net.4 (forward, dX, dW), attention and its backward, the Tree-LSTM gates, GELU and
 *     GELU', the loss and the statistics.  Activations and gradients are stored in fp32; the bf16 values exist only as
 *     operands inside the products.
 * fl_policy_forward_train_bf16 is the training forward alone (signature of fl_policy_forward_f32, this workspace): its
 * logits and values are bit-identical to those fl_policy_ppo_grad_bf16 writes for the same weights and observations. */
size_t fl_policy_workspace_bytes_grad_bf16(int64_t n_agents_total);
int fl_policy_ppo_grad_bf16(const float *const *d_weights, void *d_workspace, size_t workspace_bytes, int64_t E, int64_t N,
                            const float *d_agent_attr, const float *d_forest, const int32_t *d_adjacency,
                            const int32_t *d_node_order, const uint8_t *d_valid_actions,
                            const uint8_t *d_actions, const float *d_old_log_probs,
                            const float *d_advantages, const float *d_returns,
                            const uint8_t *d_acted,
                            const FlPpoParams *params,
                            float *const *d_grads,
                            float *d_logits, float *d_value, float *d_stats, void *stream);
int fl_policy_forward_train_bf16(const float *const *d_weights, void *d_workspace, size_t workspace_bytes, int64_t E, int64_t N,
                                 const float *d_agent_attr, const float *d_forest, const int32_t *d_adjacency,
                                 const int32_t *d_node_order, float *d_logits, float *d_value, void *stream);

/* Data-parallel learning: one minibatch split by rows into shards (one per GPU), each shard's loss divided by the counts of
 * the whole minibatch, so that the shard gradients sum to the minibatch's gradient.
 *
 * fl_policy_ppo_counts writes d_counts [2] i64 = [|S|, acted rows] of these E rows (S and rows as in the loss statement of
 * fl_policy_ppo_grad_f32), computed from d_valid_actions [E][N][5] u8 and d_acted [E] u8 alone.  Integer counts: their sum
 * over shards, in any order, is the minibatch's count.  One memset and one kernel on `stream`, no host synchronisation.
 *
 * fl_policy_ppo_grad_shard_f32 / _bf16 take the arguments of fl_policy_ppo_grad_f32 / _bf16 and d_global_counts, a device
 * pointer to [|S_g|, rows_g] i64: |S| and the acted rows of the whole minibatch (the sum over its shards of
 * fl_policy_ppo_counts), read on the device.  With S, rows the sets of this shard, the shard's loss is
 *   L_shard = sum_S( -min(r A, clip(r, 1 - clip_eps, 1 + clip_eps) A) ) / |S_g| - ent_coef sum_S(H) / |S_g|
 *             + vf_coef sum_rows((V - R)^2) / rows_g,
 * a term with a zero denominator contributing 0; every symbol, the tie rule and the arithmetic are those of
 * fl_policy_ppo_grad_f32 / _bf16.  The sum over the shards of L_shard is L of the whole minibatch, so:
 *   - d_grads: dL_shard / dparameter, this shard's contribution; the sum over shards is dL/dparameter of the minibatch.
 *   - d_stats [8]: entries 0..4 and 7 are this shard's sums over S (over rows for entry 1) divided by |S_g| (rows_g), so
 *     their sum over shards is the minibatch's statistic; entries 5 and 6 are |S| and the acted rows of this shard, so
 *     their sum is the minibatch's count.
 *   - d_logits, d_value: as fl_policy_ppo_grad_f32 / _bf16; they do not depend on the counts.
 * Given d_global_counts = fl_policy_ppo_counts of its own rows, a shard call writes the bytes fl_policy_ppo_grad_f32 / _bf16
 * write (those calls are this path with the counts taken from the workspace).  The training forward, the backward, the
 * determinism and the one host synchronisation are those calls'.  FL_ERR_BAD_ARG before any CUDA call for the argument
 * errors of fl_policy_ppo_grad_f32 and for a NULL d_global_counts; for fl_policy_ppo_counts, for a NULL pointer, E <= 0,
 * N <= 0, or E N above the 32-bit node-id bound of fl_policy_ppo_grad_f32. */
int fl_policy_ppo_counts(int64_t E, int64_t N, const uint8_t *d_valid_actions, const uint8_t *d_acted, int64_t *d_counts,
                         void *stream);
int fl_policy_ppo_grad_shard_f32(const float *const *d_weights, void *d_workspace, size_t workspace_bytes, int64_t E, int64_t N,
                                 const float *d_agent_attr, const float *d_forest, const int32_t *d_adjacency,
                                 const int32_t *d_node_order, const uint8_t *d_valid_actions,
                                 const uint8_t *d_actions, const float *d_old_log_probs,
                                 const float *d_advantages, const float *d_returns,
                                 const uint8_t *d_acted, const int64_t *d_global_counts,
                                 const FlPpoParams *params,
                                 float *const *d_grads,
                                 float *d_logits, float *d_value, float *d_stats, void *stream);
int fl_policy_ppo_grad_shard_bf16(const float *const *d_weights, void *d_workspace, size_t workspace_bytes, int64_t E, int64_t N,
                                  const float *d_agent_attr, const float *d_forest, const int32_t *d_adjacency,
                                  const int32_t *d_node_order, const uint8_t *d_valid_actions,
                                  const uint8_t *d_actions, const float *d_old_log_probs,
                                  const float *d_advantages, const float *d_returns,
                                  const uint8_t *d_acted, const int64_t *d_global_counts,
                                  const FlPpoParams *params,
                                  float *const *d_grads,
                                  float *d_logits, float *d_value, float *d_stats, void *stream);

/* Options of the PPO loss: clipped value loss and advantage normalisation over the whole minibatch.  Every symbol (S, rows, A,
 * R, V, r, the tie rule, the arithmetic) is that of fl_policy_ppo_grad_f32, and for a shard that of fl_policy_ppo_grad_shard_*.
 *   - norm_adv = 1: A_S = the row advantage listed once per agent of S (the set the policy term averages over), of the whole
 *     minibatch: n = |S_g|, and the float64 sums sum_S A, sum_S A^2 of all its shards.  mu = sum A / n; sigma = the unbiased
 *     standard deviation, sqrt(max(0, (sum A^2 - (sum A)^2 / n) / (n - 1))), 0 when n < 2 (torch's A_S.std()).  Then
 *       A_hat = (A - mu) / (sigma + adv_eps),  0 where sigma + adv_eps = 0,
 *     formed in float64 and rounded once to fp32, replaces A everywhere in the policy term and in its statistics.
 *   - vf_clip > 0: V_old = d_old_values [E] f32, the behaviour critic's value of the row, V_clip = V_old + clip(V - V_old,
 *     -vf_clip, vf_clip), and the value term becomes vf_coef mean_rows(max((V - R)^2, (V_clip - R)^2)).  d/dV = 2 (V - R)
 *     where (V - R)^2 >= (V_clip - R)^2, ties included, and 0 otherwise: exact, since the clipped square can only be strictly
 *     larger when V lies outside the band, where V_clip does not depend on V.  Statistic 1 is the mean of that max term and
 *     statistic 7 is L; the other statistics keep their meaning.
 * vf_clip < 0 or NaN, norm_adv other than 0 and 1, adv_eps < 0 or not finite: FL_ERR_BAD_ARG. */
typedef struct FlPpoOptions {
    float   vf_clip;    /* > 0: clipped value loss with this half-width; 0: off */
    int32_t norm_adv;   /* 1: normalise advantages over S of the whole minibatch; 0: off */
    float   adv_eps;    /* >= 0 and finite */
} FlPpoOptions;

/* fl_policy_ppo_moments writes d_moments [2] f64 = [sum_S A, sum_S A^2] of these E rows (d_advantages [E] f32; S from
 * d_valid_actions and d_acted as in fl_policy_ppo_counts).  One kernel on `stream` (one CTA, a fixed-order reduction, no
 * atomics: the same inputs give the same bytes), no host synchronisation.  Argument errors as fl_policy_ppo_counts. */
int fl_policy_ppo_moments(int64_t E, int64_t N, const uint8_t *d_valid_actions, const uint8_t *d_acted, const float *d_advantages,
                          double *d_moments, void *stream);

/* fl_policy_ppo_grad_ex_f32 / _bf16: fl_policy_ppo_grad_shard_f32 / _bf16 with the options above, arguments in the same order
 * plus d_old_values (may be NULL when vf_clip == 0), d_global_moments ([sum_S A, sum_S A^2] f64 of the whole minibatch, the
 * sum over its shards of fl_policy_ppo_moments, read on the device) and opts.
 *   - d_global_counts NULL: these rows are the whole minibatch and their counts are computed in the workspace, as
 *     fl_policy_ppo_grad_f32 / _bf16 do.  d_global_moments NULL likewise: the moments of these rows, computed in the
 *     workspace.  d_global_moments is not read when norm_adv = 0.
 *   - With vf_clip = 0 and norm_adv = 0 a call writes the bytes of fl_policy_ppo_grad_f32 / _bf16 (d_global_counts NULL) or
 *     of fl_policy_ppo_grad_shard_f32 / _bf16, with the same launches: those four calls are this path with the options off.
 *   - norm_adv = 1 with d_global_moments NULL adds one single-CTA launch (the moments); vf_clip adds none.  The workspace
 *     size, the determinism and the one host synchronisation are those of fl_policy_ppo_grad_f32.
 * FL_ERR_BAD_ARG before any CUDA call for the argument errors of fl_policy_ppo_grad_f32, a NULL opts, a bad option, a NULL
 * d_old_values with vf_clip > 0, and d_global_moments without d_global_counts. */
int fl_policy_ppo_grad_ex_f32(const float *const *d_weights, void *d_workspace, size_t workspace_bytes, int64_t E, int64_t N,
                              const float *d_agent_attr, const float *d_forest, const int32_t *d_adjacency,
                              const int32_t *d_node_order, const uint8_t *d_valid_actions,
                              const uint8_t *d_actions, const float *d_old_log_probs,
                              const float *d_advantages, const float *d_returns,
                              const uint8_t *d_acted, const int64_t *d_global_counts,
                              const FlPpoParams *params,
                              float *const *d_grads,
                              float *d_logits, float *d_value, float *d_stats, void *stream,
                              const float *d_old_values, const double *d_global_moments, const FlPpoOptions *opts);
int fl_policy_ppo_grad_ex_bf16(const float *const *d_weights, void *d_workspace, size_t workspace_bytes, int64_t E, int64_t N,
                               const float *d_agent_attr, const float *d_forest, const int32_t *d_adjacency,
                               const int32_t *d_node_order, const uint8_t *d_valid_actions,
                               const uint8_t *d_actions, const float *d_old_log_probs,
                               const float *d_advantages, const float *d_returns,
                               const uint8_t *d_acted, const int64_t *d_global_counts,
                               const FlPpoParams *params,
                               float *const *d_grads,
                               float *d_logits, float *d_value, float *d_stats, void *stream,
                               const float *d_old_values, const double *d_global_moments, const FlPpoOptions *opts);

/* One tensor-core product of fl_policy_ppo_grad_bf16, exposed for tests.  bf16-rounded operands, fp32 accumulation; every
 * other term in fp32.  X(m, k) = x1[row(m) ldx1 + k] (k < K1), x2[m ldx2 + k - K1] (K1 <= k < K = K1 + K2); row(m) = idx ?
 * idx[m] : m.  Row strides in floats.
 *   FL_TC_FORWARD  c[m][n] (ldc) = act(sum_k X(m, k) w[n][k] + bias[n]), m < M, n < N; w is [N][K]; pre (optional) gets
 *                  the value before the activation at c's offsets; act 0 none, 1 GELU(erf).
 *   FL_TC_DX       c[r(m)][k] = (sum_n dy[m][n] w[n][k] + add[m][k] + accum c[r(m)][k]) * gelu'(gpre[m][k]), k < K, n < N;
 *                  w is [N][ldw]; r(m) = cidx ? cidx[m] : m; add, gpre optional.
 *   FL_TC_DW       c[n][k] (row stride K) = sum over m < M of dy[m][n] X(m, k), db[n] (optional) = sum of dy[m][n]; over
 *                  fixed row chunks into d_workspace (at least 512 rows each, at most 128 chunks: 4 nch N (K + 1) bytes).
 * FL_ERR_BAD_ARG for a NULL operand or inconsistent sizes. */
#define FL_TC_FORWARD 0
#define FL_TC_DX 1
#define FL_TC_DW 2
typedef struct FlTcProduct {
    int32_t kind;
    int64_t M; int32_t N, K;
    const float *x1; const int32_t *idx; int64_t ldx1; int32_t K1;
    const float *x2; int64_t ldx2; int32_t K2;
    const float *dy; int64_t lddy;
    const float *w; int64_t ldw; const float *bias;
    float *c; const int32_t *cidx; int64_t ldc;
    const float *add; int64_t ldadd; int32_t accum;
    float *pre; int32_t act;
    const float *gpre; int64_t ldgpre;
    float *db;
} FlTcProduct;
int fl_policy_tc_product_bf16(const FlTcProduct *p, void *d_workspace, size_t workspace_bytes, void *stream);

/* Actor._choose_action in "soft" mode for every agent (plfActor.py:27-44): masked softmax over the valid actions,
 * then numpy's choice with the generator re-seeded to 42, i.e. the first action whose cumulative probability
 * exceeds 0.3745401188473625; no valid action -> 0.  d_valid_actions [n][5] u8, d_actions [n] u8. */
int fl_policy_choose_actions(const float *d_logits, const uint8_t *d_valid_actions, uint8_t *d_actions,
                             int64_t n_agents_total, void *stream);

/* Exploration for PPO rollouts: the same masked soft choice as fl_policy_choose_actions, with a seeded uniform per agent and
 * step in place of the fixed one (csrc/policy/rollout.cuh).  d_logits [E][N][5] f32, d_valid_actions [E][N][5] u8,
 * d_actions [E][N] u8, d_log_probs [E][N] f32.
 *
 * Uniform of agent i of row e: Philox4x32-10 (Random123 constants and round function) with
 *   counter = (step & 0xffffffff, step >> 32, env_offset + e, i),  key = (seed & 0xffffffff, seed >> 32),
 * output words x0 x1 x2 x3;  u = ((x0 >> 5) * 67108864.0 + (x1 >> 6)) / 9007199254740992.0   (53 bits, in [0, 1), float64).
 * Choice: the first valid action whose normalised cumulative probability (fp32 exponentials of logit - max over the valid
 * actions, cumulated in float64) exceeds u; no valid action -> 0.
 * log_probs: fp32 (x_a - max) - log(sum of those exponentials) of the chosen action a; 0 when no action is valid.
 * The draw depends only on (seed, step, env_offset + e, i): a shard that passes env_offset = its first global environment id
 * samples exactly what one device sampling the whole batch would.  FL_ERR_BAD_ARG before any CUDA call for a NULL pointer,
 * E <= 0, N <= 0, env_offset < 0 or env_offset + E > 2^32. */
int fl_policy_sample_actions(const float *d_logits, const uint8_t *d_valid_actions, int64_t E, int64_t N,
                             int64_t env_offset, uint64_t seed, uint64_t step,
                             uint8_t *d_actions, float *d_log_probs, void *stream);

/* Generalised advantage estimation over a rollout buffer of T steps of E environments with N agents each.
 * d_rewards [T+1][E][N] i32 and d_dones [T+1][E][N+1] u8 are the rows the batch returned (row k + 1: after step k; row 0 is
 * not read; of d_dones only column N, "__all__", is read); d_values [T+1][E] f32 the critic values of rows 0..T;
 * d_acted [T][E] u8: 0 where step k only reset an environment whose episode had ended (its action was ignored).
 * With r_k+1 = mean over agents of rewards[k+1][e][:] (the critic is a mean over agents) and d_k+1 = dones[k+1][e][N]:
 *   delta_k = r_k+1 + gamma V_k+1 (1 - d_k+1) - V_k
 *   A_k     = delta_k + gamma lam (1 - d_k+1) A_k+1,   A_T = 0,  A_k+1 as stored
 *   R_k     = A_k + V_k
 *   A_k = R_k = 0 where acted[k][e] == 0.
 * An episode that ends at its step limit is terminal (the limit is part of the environment): no bootstrap.  Float64
 * arithmetic, fp32 results d_advantages, d_returns [T][E].  One warp per environment.  FL_ERR_BAD_ARG before any CUDA call
 * for a NULL pointer or T, E, N <= 0. */
int fl_policy_gae(const int32_t *d_rewards, const uint8_t *d_dones, const float *d_values, const uint8_t *d_acted,
                  int64_t T, int64_t E, int64_t N, float gamma, float lam,
                  float *d_advantages, float *d_returns, void *stream);

/* One dense layer on the tensor-core path, exposed for tests: C[M][ldc] (bf16) = act(A[M][K] . W[N][K]^T + bias),
 * K and N multiples of 64 / 128, act 0 = none, 1 = GELU(erf). */
int fl_policy_linear(const uint16_t *d_a, int64_t lda, const uint16_t *d_w, const float *d_bias, uint16_t *d_c,
                     int64_t ldc, int64_t M, int64_t N, int64_t K, int act, void *stream);

/* Tuning only: fl_policy_linear that also writes SM-clock timestamps of CTA (0,0) into d_clocks[128]
 * ([0] MMA warp start, [1] weights resident, [2] end, [3] kernel start; [8+4t..] MMA thread per tile t < 8: accumulator
 * free, first stage full, last stage full; [48+4t..] epilogue warp 0: accumulator full, read, stored; [80+t] producer
 * starts tile t). */
int fl_policy_linear_debug(const uint16_t *d_a, int64_t lda, const uint16_t *d_w, const float *d_bias, uint16_t *d_c,
                           int64_t ldc, int64_t M, int64_t N, int64_t K, int act, long long *d_clocks, void *stream);

/* Tuning only: while set (non-NULL), k_tree_leaf of later forwards writes SM-clock stamps of its CTA 0 into d_clocks[128]. */
void fl_policy_debug_clocks(long long *d_clocks);

uint64_t fl_policy_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif

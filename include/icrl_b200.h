/*
 * icrl_b200 -- C ABI of the B200 (sm_100a) implementation of the ICRL per-iteration learner hot path.
 *
 * The reference (shehryar-malik/icrl) is pure Python and has no FFI layer; its boundary for this path
 * is the Python API of ConstraintNet / RolloutBufferWithCost / PPOLagrangian.  Each entry point below
 * names the reference function it replaces (file:line under /root/reference).  The Python host side
 * (icrl_b200/*.py) binds these with ctypes and keeps the reference's class / method signatures; a
 * maintainer of the reference would bind them the same way (see INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types.  `stream` is a cudaStream_t passed as void*
 *     (NULL = the legacy default stream).  Device-pointer entry points only enqueue work on `stream`
 *     (no host synchronisation) unless stated; `*_host` entry points take HOST buffers, do the H2D /
 *     D2H copies themselves on `stream` and return after synchronising it (they are the end-to-end path
 *     the reference-facing methods with numpy arguments call).
 *   - every function returns 0 on success, a positive cudaError_t value on a CUDA failure, or a
 *     negative ICRL_E* code on a bad argument.  icrl_last_error() gives a human readable message.
 *   - all floating point data is float32 unless the name says f64.  Matrices are row-major.
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef ICRL_B200_H
#define ICRL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ICRL_ABI_VERSION 2

#define ICRL_EINVAL (-1)      /* bad argument (message in icrl_last_error) */
#define ICRL_EUNSUPPORTED (-2) /* shape outside what the kernels were built for */
#define ICRL_EPEER (-3)        /* data-parallel mode: a peer rank did not deliver its part of an exchange in time */

#define ICRL_MAX_SELECT 512   /* max len(select_dim) of a constraint net */
#define ICRL_MAX_HIDDEN 3     /* max number of hidden layers of a constraint net */
#define ICRL_CN_MAX_WIDTH 64  /* max hidden width of a constraint net */

int icrl_abi_version(void);
const char* icrl_last_error(void);
/* number of kernels this library has launched since load (bench.py's `gpu_launches`) */
int64_t icrl_launch_count(void);
/* device properties the host side sizes grids with; returns 0 and fills *sm_count / *cc (e.g. 100) */
int icrl_device_info(int32_t* sm_count, int32_t* cc);
/* measured arithmetic peaks of the current device in TFLOP/s (bench.py's compute rooflines; synchronous, ~50 ms):
 * tflops2[0] = FP32 FFMA, tflops2[1] = mma.sync.m16n8k8 TF32 with fp32 accumulate (K4 issues three per fp32-class product) */
int icrl_measure_peaks(double* tflops2, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Constraint net description (ConstraintNet.__init__ state, icrl/constraint_net.py:15-99).
 * `select[i]` indexes concat([obs (obs_dim), acs (acs_dim, one-hot when is_discrete)]) exactly as
 * ConstraintNet.select_dim does (constraint_net.py:87-99, 272-273).  `params` is the flat float32
 * vector [W0 (h1 x n_select), b0, W1, b1, ..., W_out (1 x h_last), b_out] == network.state_dict() order.
 * obs_mean / obs_rstd are float64 (the reference normalises in float64, constraint_net.py:275-283);
 * obs_rstd[i] = 1 / sqrt(obs_var[i] + eps).
 */
typedef struct icrl_cn_desc {
    int32_t obs_dim;
    int32_t acs_dim;
    int32_t is_discrete;
    int32_t n_select;
    int32_t select[ICRL_MAX_SELECT];
    int32_t n_hidden;
    int32_t hidden[ICRL_MAX_HIDDEN];
    int32_t has_norm;        /* obs_mean / obs_rstd are valid */
    int32_t has_clip_obs;    /* clip obs to +-clip_obs after normalisation */
    int32_t has_clip_acs;    /* clip continuous actions to [acs_low, acs_high] */
    double clip_obs;
    const float* params;     /* device */
    const double* obs_mean;  /* device [obs_dim] or NULL */
    const double* obs_rstd;  /* device [obs_dim] or NULL */
    const float* acs_low;    /* device [acs_dim] or NULL */
    const float* acs_high;   /* device [acs_dim] or NULL */
} icrl_cn_desc;

int64_t icrl_cn_param_count(const icrl_cn_desc* d);

/* K1 -- replaces ConstraintNet.cost_function / prepare_data / forward (constraint_net.py:121-130,
 * 258-299, 101-119) for a whole batch of rows (the relabel form of VecCostWrapper.step_wait,
 * vec_cost_wrapper.py:51-66).  obs is [n_rows, obs_dim] float32 or float64 (obs_is_f64), acs is
 * [n_rows, acs_dim] float32 ([n_rows] or [n_rows,1] action indices stored as float32 when is_discrete).
 * out[n_rows] = 1 - zeta(x) when out_kind == 0 (cost), zeta(x) when out_kind == 1 (prediction). */
int icrl_cn_forward(const icrl_cn_desc* d, const void* obs, int32_t obs_is_f64, const float* acs,
                    int64_t n_rows, float* out, int32_t out_kind, void* stream);
/* same with HOST buffers (obs, acs, out); synchronous.  This is the per-environment-step call of
 * VecCostWrapper.step_wait (vec_cost_wrapper.py:62): batches of up to 64 KB are copied into one host-mapped pinned block that
 * the kernel reads and writes directly (one launch + one synchronisation; <= 16 rows run a CTA-per-row kernel); larger batches
 * are staged through device scratch. */
int icrl_cn_forward_host(const icrl_cn_desc* d, const void* obs, int32_t obs_is_f64, const float* acs,
                         int64_t n_rows, float* out, int32_t out_kind, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K2 -- replaces ConstraintNet.train + compute_is_weights + ConstraintNet.get + th.optim.Adam.step
 * (constraint_net.py:137-256, 301-317): full batch (batch_size None, what the shipped configs use) or minibatches
 * (`-cbs`): one numpy permutation of min(n_nominal, n_expert) per backward iteration, the SAME batch indices into the
 * nominal and the expert set, one Adam step per minibatch, importance weights from the full nominal set.
 */
typedef struct icrl_cn_train_cfg {
    int32_t iterations;              /* backward_iters */
    int32_t importance_sampling;     /* !no_importance_sampling */
    int32_t per_step_is;             /* per_step_importance_sampling (reproduces the reference's broadcast, quirk A) */
    int32_t train_gail_lambda;       /* BCE variant (constraint_net.py:193-197) */
    float eps;                       /* ConstraintNet.eps (1e-5) */
    float regularizer_coeff;
    float target_kl_old_new;         /* -1 disables */
    float target_kl_new_old;         /* -1 disables */
    double lr;                       /* already evaluated lr_schedule(progress) */
    double adam_beta1, adam_beta2, adam_eps;
    int32_t batch_size;              /* 0: full batch (cn_batch_size None); > 0: minibatch size (constraint_net.py:304-317) */
    const int32_t* perm;             /* batch_size > 0: device int32 [iterations][min(n_nominal, n_expert)], the permutations
                                        numpy would draw (constraint_net.py:306) -- generated by the host so seeds stay compatible */
} icrl_cn_train_cfg;

/* metrics written by icrl_cn_train (host struct), the `backward/ *` keys of constraint_net.py:209-227 */
typedef struct icrl_cn_train_metrics {
    float cn_loss, expert_loss, unweighted_nominal_loss, nominal_loss, regularizer_loss;
    float is_mean, is_max, is_min;
    float nominal_preds_max, nominal_preds_min, nominal_preds_mean;
    float expert_preds_max, expert_preds_min, expert_preds_mean;
    float kl_old_new, kl_new_old;
    int32_t early_stop_itr;
    int32_t steps_taken;             /* Adam steps actually applied */
} icrl_cn_train_metrics;

/* d->params is updated in place (cast away const); adam_m / adam_v are [param_count] device float32,
 * *adam_step (host int64) is read and advanced.  nominal/expert obs+acs are device arrays as for K1;
 * episode_offsets is a device int32 [n_episodes+1] prefix sum of episode_lengths.  Synchronous (returns
 * metrics).  Workspace is allocated internally and cached. */
int icrl_cn_train(const icrl_cn_desc* d, const icrl_cn_train_cfg* cfg,
                  const void* nominal_obs, int32_t nominal_obs_is_f64, const float* nominal_acs, int64_t n_nominal,
                  const int32_t* episode_offsets, int32_t n_episodes,
                  const void* expert_obs, int32_t expert_obs_is_f64, const float* expert_acs, int64_t n_expert,
                  float* adam_m, float* adam_v, int64_t* adam_step,
                  icrl_cn_train_metrics* metrics, void* stream);

/* Data-parallel K2 across the GPUs of one node (SURVEY section 8(e): "shard nominal rows by whole episodes and expert rows
 * evenly").  Every rank passes ITS nominal episodes / expert rows to the same call; the partial sums of the three reductions of
 * a backward iteration (sum of IS ratios + per-episode products; sum / max / min of the weights; gradient + loss sums) are
 * stored by the kernels straight into every rank's exchange buffer (icrl_comm_alloc'ed, CUDA-IPC mapped, NVLink peer stores),
 * published with a per-exchange sequence flag and summed in rank order by the consuming kernel, so all replicas apply
 * bit-identical Adam steps.  No host synchronisation inside, no NCCL.  Returns ICRL_EPEER when a peer did not deliver within
 * ~2 s.  Minibatch mode is not available here (ICRL_EUNSUPPORTED). */
typedef struct icrl_cn_dist {
    int32_t rank, world;
    void* recv[8];                   /* recv[r]: rank r's exchange buffer (>= icrl_cn_dist_bytes), recv[rank] is local; zeroed at allocation */
    int64_t buffer_bytes;            /* size of each exchange buffer */
    uint32_t seq_base;               /* every rank advances it by iterations + 1 after each call */
    int64_t n_nominal_global, n_expert_global;   /* row counts over all ranks (the loss means divide by these) */
    int32_t n_episodes_global, episode_base;     /* episodes over all ranks; global index of this rank's first episode */
} icrl_cn_dist;
int64_t icrl_cn_dist_bytes(const icrl_cn_desc* d, int32_t n_episodes_global);
int icrl_cn_train_dist(const icrl_cn_desc* d, const icrl_cn_train_cfg* cfg,
                       const void* nominal_obs, int32_t nominal_obs_is_f64, const float* nominal_acs, int64_t n_nominal,
                       const int32_t* episode_offsets, int32_t n_episodes,
                       const void* expert_obs, int32_t expert_obs_is_f64, const float* expert_acs, int64_t n_expert,
                       float* adam_m, float* adam_v, int64_t* adam_step,
                       icrl_cn_train_metrics* metrics, const icrl_cn_dist* dist, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K3 -- replaces RolloutBufferWithCost.compute_returns_and_advantage (both calls of
 * _compute_returns_and_advantage, stable_baselines3/common/buffers.py:493-552).  All [T,E] arrays are
 * time-major float32 as the buffer stores them (buffers.py:468-491); last_dones is [E] uint8 (numpy bool).
 * The running advantage is carried in float64 as the reference does (numpy promotion of `1.0 - bool`). */
int icrl_dual_gae(const float* rewards, const float* reward_values, const float* costs, const float* cost_values,
                  const float* dones, const float* reward_last_value, const float* cost_last_value,
                  const uint8_t* last_dones, int32_t T, int32_t E,
                  double reward_gamma, double reward_gae_lambda, double cost_gamma, double cost_gae_lambda,
                  float* reward_advantages, float* reward_returns, float* cost_advantages, float* cost_returns,
                  void* stream);
/* HOST buffers; synchronous (rollout-sized buffers, <= 1 MB in total, run on a host-mapped pinned block). */
int icrl_dual_gae_host(const float* rewards, const float* reward_values, const float* costs, const float* cost_values,
                       const float* dones, const float* reward_last_value, const float* cost_last_value,
                       const uint8_t* last_dones, int32_t T, int32_t E,
                       double reward_gamma, double reward_gae_lambda, double cost_gamma, double cost_gae_lambda,
                       float* reward_advantages, float* reward_returns, float* cost_advantages, float* cost_returns,
                       void* stream);

/* ------------------------------------------------------------------------------------------------
 * K4 -- replaces the epoch / minibatch loop of PPOLagrangian.train (stable_baselines3/ppo_lag/ppo_lag.py:
 * 198-297): ActorTwoCriticsPolicy.evaluate_actions (common/policies.py:752-767), the clipped surrogate +
 * nu * cost term, both value losses, entropy, backward, clip_grad_norm_, Adam -- for every minibatch of
 * every epoch in ONE persistent launch, with the per-epoch target_kl early stop evaluated on the device.
 *
 * Policy: three separate tanh MLP trunks obs -> h0 -> h1 (pi, vf, cvf; torch_layers.py:129-254), each with its own
 * {h0, h1} (`trunk_hidden`, or `hidden` for all three), and linear heads on their own trunk's last layer.  `params` /
 * `adam_m` / `adam_v` are flat float32 device vectors in the reference's parameters() order: [log_std (act_dim,
 * continuous only)], then for each trunk t of pi, vf, cvf: W0 (h0[t] x obs_dim), b0, W1 (h1[t] x h0[t]), b1; then
 * action_net W (act_out x h1[pi]), b; value_net W (1 x h1[vf]), b; cost_value_net W (1 x h1[cvf]), b.
 *
 * Rollout data are device arrays in the buffer's TIME-MAJOR layout [T, E, ...]; minibatch indices in
 * `perm` refer to the reference's env-major flattening (row = e*T + t, buffers.py:52-65,598-603) and are
 * translated on the device, so no transposed copy is ever made.  `perm` is int32 [n_epochs, T*E]: the
 * permutations numpy would draw (buffers.py:596), generated by the host so seeds stay compatible.
 *
 * Two regimes behind the same entry point (the reference allows any batch_size, None = the whole buffer, buffers.py:605-607):
 *   batch_size <  2048  one persistent 6-CTA cluster (a CTA pair per trunk) runs all epochs: the dependent-step latency regime
 *                       of the shipped configs (64 / 128 rows x 1 600 steps per rollout);
 *   batch_size >= 2048  "wide": as many 6-CTA clusters as fit the device (24 on a B200) share every minibatch, one launch per
 *                       epoch; per optimiser step the clusters' gradients are summed in cluster order through L2 between two
 *                       grid-wide barriers and every cluster applies the same clip + Adam step to its replica.
 * ICRL_PPO_WIDE=0/1 forces the choice, ICRL_PPO_WIDE_CLUSTERS=n the cluster count (tests).
 */
typedef struct icrl_ppo_cfg {
    int32_t obs_dim, act_dim, is_discrete; /* act_dim = action dims (continuous) or number of actions (discrete) */
    int32_t hidden[2];
    int32_t T, E;
    int32_t batch_size, n_epochs;
    int32_t has_target_kl, has_clip_vf_reward, has_clip_vf_cost;
    float clip_range, clip_range_reward_vf, clip_range_cost_vf;
    float ent_coef, reward_vf_coef, cost_vf_coef, max_grad_norm, target_kl;
    float nu;                               /* current penalty self.dual.nu().item() (ppo_lag.py:234) */
    double lr, adam_beta1, adam_beta2, adam_eps;
    int32_t max_steps;                      /* >0: stop after that many optimiser steps (bench sampling); 0 = all */
    int32_t trunk_hidden[3][2];             /* {h0, h1} of the pi, vf and cvf trunks, each in 1..64; all zeros: every trunk
                                               uses hidden[] (so zero-initialising callers keep the shared widths).  When
                                               set, hidden[] is ignored.  Appended without an ABI version change. */
} icrl_ppo_cfg;

typedef struct icrl_ppo_data {
    const float* observations;      /* [T,E,obs_dim] (normalised obs, buffer.observations) */
    const float* actions;           /* [T,E,act_dim] continuous, or [T,E,1] action index as float (discrete) */
    const float* old_log_prob;      /* [T,E] */
    const float* old_reward_values; /* [T,E] */
    const float* reward_advantages; /* [T,E] */
    const float* reward_returns;    /* [T,E] */
    const float* old_cost_values;   /* [T,E] */
    const float* cost_advantages;   /* [T,E] */
    const float* cost_returns;      /* [T,E] */
    const int32_t* perm;            /* [n_epochs, T*E] */
    const float* nu_device;         /* optional: read the penalty nu from this device float instead of cfg->nu
                                       (lets a device-resident dual state feed the next launch without a host read) */
} icrl_ppo_data;

#define ICRL_PPO_STATS_PER_STEP 8
/* per optimiser step, written to `step_stats` [n_epochs * steps_per_epoch, 8] device float32:
 * 0 policy_loss (pg_losses), 1 clip_fraction, 2 reward_value_loss, 3 cost_value_loss, 4 entropy_loss,
 * 5 approx_kl, 6 total loss, 7 grad-norm before clipping.  `result` is device int32[4]:
 * [0] early_stop_epoch (== n_epochs when no early stop), [1] optimiser steps taken, [2] != 0: an exchange wait inside the
 * kernel hit its bound (lost cluster peer / data-parallel rank; the parameters of this call are not valid), [3] internal. */
int64_t icrl_ppo_param_count(const icrl_ppo_cfg* cfg);
int icrl_ppo_train(const icrl_ppo_cfg* cfg, const icrl_ppo_data* data, float* params, float* adam_m, float* adam_v,
                   int64_t adam_step_before, float* step_stats, int32_t* result, void* stream);


/* ------------------------------------------------------------------------------------------------
 * Data-parallel K4 across the GPUs of one node (one process per GPU; SURVEY section 8(e)).  Every rank owns the rollout
 * of its own environments and runs the same persistent kernel on `batch_size` LOCAL rows per optimiser step; the
 * gradients of the three trunks are summed across ranks INSIDE the kernel: each CTA stores its gradient fragments
 * straight into the peers' receive buffers over NVLink (CUDA IPC mapped memory) as self-validating 16-byte words (no
 * fence, no separate flag), polls its own buffer and adds the contributions in rank order, so all ranks apply bit-identical
 * Adam updates and the replicated parameters never drift.  Exchange schemes (ICRL_PPO_DIST_MODE overrides the choice):
 * 2 / 4 ranks one-hop broadcast of {f0, f1, f2, seq ^ hash} words + rank-ordered sum; 8 ranks reduce-scatter + all-gather
 * with the same words; other world sizes {value, seq, value, seq} words.  The three layouts share the receive buffer.
 * The global-minibatch advantage statistics (ppo_lag.py:218-222) are data-only, so the caller
 * all-reduces one small table up front (icrl_ppo_local_advsums -> NCCL all-reduce -> icrl_ppo_dist.advsums).
 */
#define ICRL_PPO_MAX_RANKS 8
#define ICRL_PPO_RECV_BYTES (32 * 1024 * 1024) /* covers the largest receive layout: the four single-cluster layouts (<= 14.2 MB, k4_common.cuh) and the
                                                   many-cluster one [parity 2][src 8][CTA 192][2 words][256 threads] x 16 bytes = 25.2 MB */
#define ICRL_PPO_FLAG_BYTES (2 * ICRL_PPO_MAX_RANKS * 4 * 4)             /* [parity][src][trunk] uint32 */

int icrl_comm_alloc(int64_t bytes, void** dev_ptr, unsigned char* handle64);   /* zeroed device buffer + its IPC handle */
int icrl_comm_open(const unsigned char* handle64, void** dev_ptr);              /* map a peer's buffer */
int icrl_comm_close(void* dev_ptr);
int icrl_comm_free(void* dev_ptr);

typedef struct icrl_ppo_dist {
    int32_t rank, world;
    float* recv[ICRL_PPO_MAX_RANKS];       /* recv[r]: rank r's receive buffer (ICRL_PPO_RECV_BYTES); recv[rank] is local */
    uint32_t* flags[ICRL_PPO_MAX_RANKS];   /* flags[r]: rank r's flag array (ICRL_PPO_FLAG_BYTES) */
    uint32_t flag_base;                    /* monotonically growing; every rank advances it by steps+1 after each launch */
    const double* advsums;                 /* device [n_epochs*steps_per_epoch][4]: all-reduced sum adv_r, sum adv_r^2,
                                              sum adv_c, row count of every global minibatch */
} icrl_ppo_dist;

/* local partial sums of the table above for this rank's rows (to be summed over ranks by the caller) */
int icrl_ppo_local_advsums(const icrl_ppo_cfg* cfg, const icrl_ppo_data* data, double* advsums_out, void* stream);
/* icrl_ppo_train with the in-kernel gradient all-reduce; the per-step stats are global already (the loss sums ride along
 * with the gradient exchange); result[2] != 0 reports a peer time-out. */
int icrl_ppo_train_dist(const icrl_ppo_cfg* cfg, const icrl_ppo_data* data, float* params, float* adam_m, float* adam_v,
                        int64_t adam_step_before, float* step_stats, int32_t* result, const icrl_ppo_dist* dist,
                        void* stream);

/* Policy forward for rollout collection / evaluation (policies.py:716-731 without sampling):
 * head [n, act_out] (action mean or logits), values [n], cost_values [n]; obs is [n, obs_dim] row-major. */
int icrl_policy_forward(const icrl_ppo_cfg* cfg, const float* params, const float* obs, int64_t n,
                        float* head, float* values, float* cost_values, void* stream);

/* Dual variable -- replaces DualVariable.update_parameter + Nu.clamp (stable_baselines3/common/dual_variable.py:
 * 27-29,47-57) and the np.mean(rollout_buffer.orig_costs) feeding it (ppo_lag.py:303-306).  `state` is device
 * float32[6] = {log_nu, adam exp_avg, adam exp_avg_sq, last loss, nu = softplus(log_nu) after the step, mean cost};
 * the first three are read and updated, the rest written.  orig_costs is device float32 [n].  Adam uses the
 * reference's defaults for this optimiser (betas 0.9/0.999, eps 1e-8); adam_step_before counts previous updates. */
int icrl_dual_update(float* state, const float* orig_costs, int64_t n, double alpha, double lr, int64_t adam_step_before,
                     double clamp_min_log_nu, void* stream);

/* Whole-rollout cost normalisation (SURVEY 8 (f1)) -- replaces, for a [T, E] rollout relabelled by icrl_cn_forward,
 * the T per-step host updates of VecNormalizeWithCost.step_wait / _update_cost / normalize_cost
 * (stable_baselines3/common/vec_env/vec_normalize.py:232-257) and RunningMeanStd.update
 * (stable_baselines3/common/running_mean_std.py:19-39).  All device pointers.
 *   orig_costs [T, E] float32   what the cost function returned at each step
 *   dones      [T, E] float32   buffer layout: dones[t] = episode ended at step t-1 (buffers.py add());
 *   last_dones [E]    uint8     episode ended at step T-1            -> `news` of step t = dones[t+1] / last_dones
 *   state      float64 [3 + E]  {cost_rms.mean, cost_rms.var, cost_rms.count, cost_ret[E]}, read and updated when
 *                               `training` (bit-exact with the numpy float64 arithmetic, pairwise sums included)
 *   costs      [T, E] float32   clip(orig / sqrt(var_after_step_t + epsilon), +-clip_cost) when `norm_cost`, else a copy
 * (may alias orig_costs). */
int icrl_cost_normalize(const float* orig_costs, const float* dones, const uint8_t* last_dones, int32_t T, int32_t E,
                        double cost_gamma, double epsilon, double clip_cost, int32_t norm_cost, int32_t training,
                        double* state, float* costs, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ICRL_B200_H */

/*
 * openrl_b200.h — C-ABI of libopenrl_b200.so (hand-written sm_100a CUDA).
 *
 * Drop-in boundary for OpenRL's rollout-collection + PPO/MAPPO-update hot path.
 * The reference has no FFI: its seams are Python constructor-injection points
 * (SURVEY.md §8b).  Every entry point below replaces the inner loop of one
 * reference function; the Python host package `openrl_b200` binds them with ctypes
 * (openrl_b200/lib.py) and INTEGRATION.md shows the stub a reference maintainer
 * would add.
 *
 * Conventions
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless the
 *     name ends in _host; the caller owns all memory (torch tensors in practice);
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*);
 *   - return value: 0 = ok, otherwise a cudaError_t or ORL_ERR_*; the message is
 *     available from orl_last_error();
 *   - all floating-point buffers are float32, row-major, laid out like the
 *     reference's ReplayData arrays with the (env, agent) axes flattened:
 *     element (t, n, a, k) of a (T[+1], N, A, K) array is at ((t*N + n)*A + a)*K + k;
 *     B = N*A is the number of "rows" (columns of the time scan).
 */
#ifndef OPENRL_B200_H
#define OPENRL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ORL_ABI_VERSION 1

#define ORL_ERR_BAD_ARG 10001
#define ORL_ERR_UNSUPPORTED 10002

/* library / device --------------------------------------------------------------- */
int orl_abi_version(void);
const char* orl_last_error(void);
/* number of SMs of the current device (grids are sized from it) */
int orl_device_sm_count(int* sm_count_out);

/* ---- GAE / returns ---------------------------------------------------------------
 * Replaces ReplayData.compute_returns (openrl/buffers/replay_data.py:320-423, all 8
 * branches) and, fused behind it, the advantage construction of
 * PPOAlgorithm.train_ppo (openrl/algorithms/ppo.py:384-399) plus the moments needed
 * by its normalisation (ppo.py:402-409) and by ValueNorm.update on a full-buffer
 * minibatch (openrl/modules/utils/valuenorm.py:59-76).
 *
 * flags: */
#define ORL_GAE_USE_GAE 1            /* cfg.use_gae */
#define ORL_GAE_PROPER_TIME_LIMITS 2 /* cfg.use_proper_time_limits (reads bad_masks) */
#define ORL_GAE_DENORM 4             /* (use_popart|use_valuenorm) and normalizer given */
/*
 * rewards      (T,   B)   in
 * value_preds  (T+1, B)   in/out: row T is overwritten with next_value when USE_GAE
 * masks        (T+1, B)   in
 * bad_masks    (T+1, B)   in   (may be NULL unless PROPER_TIME_LIMITS)
 * active_masks (T+1, B)   in   (may be NULL: treated as all ones; only used for stats)
 * next_value   (B)        in   bootstrap value of slot T
 * vn_state     (3)        in   ValueNorm {running_mean, running_mean_sq, debiasing_term}
 *                              (valuenorm.py:27-35); required iff ORL_GAE_DENORM
 * returns      (T+1, B)   out  (row T = next_value when !USE_GAE, untouched otherwise)
 * advantages   (T,   B)   out  returns[:-1] - denorm(value_preds[:-1]); may be NULL
 * stats        (ORL_GAE_NSTATS doubles) out, may be NULL; ZEROED by the call, then
 *              accumulated: see ORL_GS_* indices.
 * gamma, gae_lambda are passed as double because the reference multiplies the two
 * Python floats in double before the product meets the float32 arrays.
 * Bit-exact with the reference's numpy float32 evaluation order (no FMA contraction).
 */
#define ORL_GAE_NSTATS 8
#define ORL_GS_ADV_SUM 0      /* sum adv            over all (t<T, b)            */
#define ORL_GS_ADV_SQSUM 1    /* sum adv^2                                        */
#define ORL_GS_COUNT 2        /* T*B                                              */
#define ORL_GS_ADV_ACT_SUM 3  /* sum adv   where active_masks[t] != 0             */
#define ORL_GS_ADV_ACT_SQSUM 4
#define ORL_GS_RET_SUM 5      /* sum returns[t<T]       } {5,6,7} is the mb_stats triple  */
#define ORL_GS_RET_SQSUM 6    /* sum returns[t<T]^2     } of orl_ppo_* for a minibatch    */
#define ORL_GS_ACT_COUNT 7    /* number of active elements } covering the whole buffer    */
int orl_gae(const float* rewards, float* value_preds, const float* masks,
            const float* bad_masks, const float* active_masks, const float* next_value,
            const float* vn_state, float* returns, float* advantages, double* stats,
            int T, int B, double gamma, double gae_lambda, int flags, void* stream);


/* ---- device-resident vectorised envs -------------------------------------------------
 * Replace SyncVectorEnv/AsyncVectorEnv stepping (openrl/envs/vec_env/sync_venv.py:129-247,
 * async_venv.py:316-430,731-875) + the per-env wrappers Single2MultiAgentWrapper /
 * RemoveTruncated (openrl/envs/wrappers/multiagent_wrapper.py:33-79,
 * extra_wrappers.py:122-134) for the simple gym-class envs.  State lives in caller-owned
 * device arrays (SoA over envs):
 *   CARTPOLE : env_f64 [4][N] (x, x_dot, theta, theta_dot) float64 like gymnasium;
 *              env_i32 [1][N] elapsed steps (TimeLimit 500);
 *              env_u64 [4][N] numpy-PCG64 {state_hi, state_lo, inc_hi, inc_lo} of the env's
 *              np_random (seeded seed + i*10086 by the host, sync_venv.py:137).
 *   GRIDWORLD: env_i32 [4][N] (x, y, steps, resets); env_table optional int32
 *              [N][env_table_len][2] start cells for parity runs; else Philox(rng_seed).
 *   NONE     : no device env (host env.step, e.g. MuJoCo): orl_rollout only acts.
 */
#define ORL_HEAD_CATEGORICAL 0
#define ORL_HEAD_GAUSSIAN 1
#define ORL_ENV_NONE 0
#define ORL_ENV_CARTPOLE 1
#define ORL_ENV_GRIDWORLD 2
#define ORL_ENV_MPE_SPREAD 3

/* Draw initial states (env.reset()) and write the observations of slot `obs_out` (B, d).
 * Mirrors SyncVectorEnv._reset (sync_venv.py:129-169).  RNG streams must already be seeded. */
int orl_env_reset(int env_kind, int n_envs, int n_agents, double* env_f64, uint64_t* env_u64,
                  int32_t* env_i32, const int32_t* env_table, int env_table_len,
                  uint64_t rng_seed, float* policy_obs_out, float* critic_obs_out, void* stream);

/* One vectorised env.step outside the fused rollout (the BaseVecEnv.step duck type used by
 * evaluation loops): actions (B) float -> obs (B,d), rewards (B), dones (B) as 0/1 floats and,
 * optionally, the pre-reset terminal observation (info["final_observation"], sync_venv.py:213-218). */
int orl_env_step(int env_kind, int n_envs, int n_agents, double* env_f64, uint64_t* env_u64,
                 int32_t* env_i32, const int32_t* env_table, int env_table_len, uint64_t rng_seed,
                 float* ep_return, int32_t* ep_length, double* episode_stats, const float* actions,
                 float* obs_out, float* rewards_out, float* dones_out, float* final_obs_out,
                 void* stream);

/* ---- fused rollout: policy forward + sampling + env.step + buffer insert -----------------
 * Replaces the body of OnPolicyDriver.actor_rollout for steps [t_begin, t_end)
 * (openrl/drivers/onpolicy_driver.py:154-203): act() :236-279 (policy half:
 * PolicyNetwork.forward_original policy_network.py:130-162, MLPBase mlp.py:160-176,
 * Categorical distributions.py:58-72, sampling = torch.multinomial == argmax(probs/q)),
 * envs.step() (see above), add2buffer() :80-152 and ReplayData.insert
 * (openrl/buffers/replay_data.py:245-284).  Envs are independent, so one launch can cover all
 * T steps (t_begin = 0, t_end = T); per-step launches (t_end = t_begin + 1) serve callbacks.
 * Critic values are produced separately by orl_critic_values (they do not influence the
 * trajectory).
 *
 * Sampling: exp_noise != NULL ("parity mode") supplies q ~ Exp(1) of shape (T, B, n) drawn by
 * the host with torch's CPU generator in the reference's order; NULL uses Philox4x32-10 keyed
 * by rng_seed with counter (rng_step_base + *rng_counter + t, row).  deterministic != 0 takes the mode.
 */
typedef struct OrlRolloutArgs {
    int32_t env_kind;       /* ORL_ENV_* */
    int32_t n_envs;         /* N */
    int32_t n_agents;       /* A; rows B = N*A */
    int32_t episode_length; /* T: depth of the (T[+1], B, .) buffers */
    int32_t t_begin, t_end; /* steps to run, 0 <= t_begin < t_end <= T */
    int32_t obs_dim;        /* d, policy observation width (<= 64) */
    int32_t critic_obs_dim; /* 0: critic obs == policy obs (critic_obs may be NULL) */
    int32_t n_actions;      /* n <= 8, Discrete(n) */
    int32_t activation_id;  /* cfg.activation_id: 0 tanh, 1 relu, 2 leaky_relu, 3 elu */
    int32_t deterministic;
    int32_t env_table_len;
    const float* policy_params; /* flat net parameters, layout in orl_mlp.cuh / DESIGN.md */
    float* policy_obs;          /* (T+1, B, d)   slot t read at t_begin, slots t+1 written */
    float* critic_obs;          /* (T+1, B, dc)  or NULL */
    float* actions;             /* (T, B, 1)  sampled index stored as float32 (replay_data.py:163-166) */
    float* action_log_probs;    /* (T, B, 1) */
    float* rewards;             /* (T, B, 1) */
    float* masks;               /* (T+1, B, 1) */
    float* active_masks;        /* (T+1, B, 1) */
    const float* action_masks;  /* (T+1, B, n) or NULL (all actions available) */
    const float* exp_noise;     /* (T, B, n) or NULL */
    uint64_t rng_seed;
    uint64_t rng_step_base;     /* Philox counter of step t is rng_step_base + *rng_counter + t */
    uint64_t* rng_counter;      /* (1) device counter or NULL; += (t_end - t_begin) after the launch,
                                   so a captured CUDA graph draws fresh noise on every replay */
    double* env_f64;
    uint64_t* env_u64;
    int32_t* env_i32;
    const int32_t* env_table;
    float* ep_return;           /* (N) running episode return  (VecMonitor-style statistics) */
    int32_t* ep_length;         /* (N) running episode length */
    double* episode_stats;      /* (4) += {sum return, sum length, #episodes, 0} of finished episodes */
    int32_t head_kind;          /* ORL_HEAD_CATEGORICAL (Discrete(n)) or ORL_HEAD_GAUSSIAN (Box(n), DiagGaussian,
                                   distributions.py:75-98): then n_actions = action width, actions and
                                   action_log_probs are (T, B, n) (per-dimension log-probs), exp_noise holds
                                   N(0,1) draws (torch.normal == noise*std + mean) and the parameter vector ends
                                   with logstd[n].  Gaussian heads act on host-stepped envs (ORL_ENV_NONE). */
    int32_t rng_row_offset;     /* added to the row index in the Philox counter: rank r of an env-sharded run passes its
                                   first global row (r * B) with the SAME rng_seed on every rank, so that sharded rollouts
                                   draw exactly the noise the unsharded run draws for those rows */
} OrlRolloutArgs;
int orl_rollout(const OrlRolloutArgs* args, void* stream);

/* ---- critic forward over a flat batch of rows ------------------------------------------
 * Replaces the critic half of act() (ValueNetwork.forward, value_network.py:113-136) for all
 * T+1 slots at once and the bootstrap forward of OnPolicyDriver.compute_returns
 * (onpolicy_driver.py:206-215).  obs (rows, d) -> values (rows). */
int orl_critic_values(const float* critic_params, int obs_dim, int activation_id,
                      const float* obs, float* values, long long rows, void* stream);

/* ---- insert of one HOST env.step into the device rollout buffer ---------------------------
 * Replaces OnPolicyDriver.add2buffer -> ReplayData.insert (onpolicy_driver.py:80-152, replay_data.py:245-284) for
 * host-stepped envs: `staged` is the step's result as ONE uploaded block [obs (B*d) | rewards (B) | dones (B)]
 * (B = n_envs * n_agents rows); writes slot t+1 of policy_obs / masks / active_masks and slot t of rewards with the
 * reference's mask rules (masks = 0 where all agents of the env are done, active_masks = 0 for a done agent of a
 * running env).  Pointers address the given slot / row range (rows of a group are contiguous). */
int orl_host_insert(const float* staged, int n_envs, int n_agents, int obs_dim, float* policy_obs_next, float* rewards,
                    float* masks_next, float* active_masks_next, void* stream);

/* ---- policy evaluation of given actions over a flat batch of rows ------------------------
 * Replaces PolicyNetwork.eval_actions (policy_network.py:164-203) -> ACTLayer.evaluate_actions (act.py:130-172), the
 * policy half of PPOModule.evaluate_actions (ppo_module.py:147-193), outside the fused update: obs (rows, d), actions
 * (rows) [Categorical: index as float32] or (rows, n) [DiagGaussian] -> log_probs and entropy with the shape of
 * `actions` (per row / per dimension; the caller takes the active-mask mean, act.py:160-168). */
int orl_policy_eval(const float* policy_params, int obs_dim, int n_actions, int activation_id, int head_kind,
                    const float* obs, const float* actions, const float* action_masks, float* log_probs,
                    float* entropy, long long rows, void* stream);


/* ---- PPO minibatch update ---------------------------------------------------------------
 * Replaces PPOAlgorithm.ppo_update (openrl/algorithms/ppo.py:46-176): prepare_loss :238-361
 * (evaluate_actions -> PolicyNetwork.eval_actions policy_network.py:164-203 / ValueNetwork.forward
 * value_network.py:113-136, ratio + clipped surrogate :300-319, cal_value_loss :178-220 incl.
 * ValueNorm.update/normalize valuenorm.py:59-90, entropy act.py:160-168, construct_loss_list
 * :226-236), loss.backward(), clip_grad_norm_ (:139-150) and Adam.step (rl_module.py:80-87), and
 * the minibatch gather of ReplayData.feed_forward_generator (replay_data.py:553-646).
 *
 * Three launches per update, all asynchronous, no host round trip:
 *   orl_ppo_fwdbwd : fused gather + forward + loss + backward over the minibatch rows; every CTA
 *                    writes its partial FOLDED gradients and loss sums to `partials`.
 *   orl_ppo_reduce : deterministic reduction of the partials over CTAs -> `folded` (2*stride
 *                    floats: policy net then critic net).  With >1 GPU the caller all-reduces
 *                    (SUM) `folded` here — the single NCCL all-reduce per update.
 *   orl_ppo_apply  : unfold to true gradients, per-net global-norm clip, Adam, ValueNorm commit,
 *                    train_info accumulation.
 * flags: */
#define ORL_PPO_HUBER 1               /* cfg.use_huber_loss */
#define ORL_PPO_CLIP_VALUE 2          /* cfg.use_clipped_value_loss */
#define ORL_PPO_VALUE_ACTIVE_MASKS 4  /* cfg.use_value_active_masks */
#define ORL_PPO_POLICY_ACTIVE_MASKS 8 /* cfg.use_policy_active_masks */
#define ORL_PPO_VALUENORM 16          /* cfg.use_valuenorm (normaliser present) */
#define ORL_PPO_ADV_NORMALIZE 32      /* cfg.use_adv_normalize (ppo.py:402-403) */
#define ORL_PPO_MAX_GRAD_NORM 64      /* cfg.use_max_grad_norm */
#define ORL_PPO_A2C 256               /* A2CAlgorithm.prepare_loss (openrl/algorithms/a2c.py:39-140): policy loss
                                         -adv * log-prob instead of the clipped surrogate; ratio reported as 0 */
#define ORL_PPO_DUAL_CLIP 512         /* cfg.dual_clip_ppo: ratio = min(ratio, dual_clip_coeff) (ppo.py:304-305) */
#define ORL_PPO_JOINT_ACTION 1024     /* cfg.use_joint_action_loss (JRPO, ppo.py:254-321): chunked recurrent update only
                                         (orl_rnn_fwdbwd, n_agents <= 4); see the JRPO layout under OrlRnnArgs.  The
                                         feed-forward entry points refuse it with ORL_ERR_UNSUPPORTED. */
#define ORL_PPO_TENSORCORE 128        /* the 64x64 GEMMs of the trunk (forward, backward-data, weight gradients) on tcgen05
                                         tensor cores with split-fp16 operands (x = hi + lo, three MMA passes, FP32
                                         accumulate in TMEM): fp32-class accuracy, same 1e-4 loss-parity bar as the FFMA
                                         kernel.  Categorical heads, obs widths <= 8, |obs| < 65504.  Minibatch tiles are
                                         staged by TMA when `indices` is NULL, by cp.async gathers otherwise.
                                         Without the flag everything is fp32 FFMA. */
#define ORL_PPO_TF32 ORL_PPO_TENSORCORE /* round-1 name of the flag */

typedef struct OrlPpoArgs {
    int32_t obs_dim;         /* d  policy obs width  (<= 64) */
    int32_t critic_obs_dim;  /* dc critic obs width  (<= 64) */
    int32_t n_actions;       /* n <= 8 */
    int32_t activation_id;
    int32_t flags;           /* ORL_PPO_* */
    int32_t grid_per_net;    /* CTAs per net in orl_ppo_fwdbwd (partials has 2*grid_per_net rows) */
    int64_t batch_rows;      /* rows of this minibatch */
    int64_t row_begin;       /* used when indices == NULL: rows [row_begin, row_begin+batch_rows) */
    int64_t total_rows;      /* T*B, rows of the flattened buffers (bounds) */
    const int64_t* indices;  /* (batch_rows) flat row ids (torch.randperm slice) or NULL */
    /* rollout data flattened to (T*B, .) */
    const float* policy_obs;     /* (T*B, d)  */
    const float* critic_obs;     /* (T*B, dc) */
    const float* actions;        /* (T*B)     */
    const float* old_log_probs;  /* (T*B)     */
    const float* advantages;     /* (T*B) raw, normalised on the fly from gae_stats */
    const float* value_preds;    /* (T*B)     */
    const float* returns;        /* (T*B)     */
    const float* active_masks;   /* (T*B)     */
    const float* action_masks;   /* (T*B, n) or NULL */
    const double* gae_stats;     /* (ORL_GAE_NSTATS) global moments of the raw advantages */
    const double* mb_stats;      /* (3) {sum returns, sum returns^2, sum active} over this minibatch */
    float* vn_state;             /* (3) ValueNorm state BEFORE this update; orl_ppo_apply commits the update */
    float* policy_params;        /* flat, updated in place by orl_ppo_apply */
    float* critic_params;
    float* policy_adam_m; float* policy_adam_v;   /* Adam moments, same layout as params */
    float* critic_adam_m; float* critic_adam_v;
    int32_t* adam_steps;         /* (2) step counters {policy, critic}, incremented by apply */
    const float* lrs;            /* (2) {lr, critic_lr} (device so that CUDA graphs can be replayed) */
    float clip_param, entropy_coef, value_loss_coef, huber_delta, max_grad_norm;
    float adam_beta1, adam_beta2, adam_eps, weight_decay;
    float reserved0;
    double vn_beta;              /* ValueNorm beta (0.99999); double: (1 - beta) is taken in double like the reference */
    float* partials;             /* (2*grid_per_net, stride) scratch */
    float* folded;               /* (2, stride): reduced folded gradients + loss sums */
    float* grads;                /* (2, orl_ppo_grads_stride): true gradients, parameter layout (written by apply) */
    float* train_info;           /* (6) += {value_loss, critic_grad_norm, policy_loss, dist_entropy,
                                             actor_grad_norm, ratio}  (ppo.py:430-451) */
    int32_t head_kind;           /* ORL_HEAD_*: with GAUSSIAN actions / old_log_probs are (T*B, n) */
    float dual_clip_coeff;       /* cfg.dual_clip_coeff (used with ORL_PPO_DUAL_CLIP) */
    int64_t norm_rows;           /* rows of the GLOBAL minibatch (all ranks): the 1/rows loss weights, the reported
                                    ratio mean and the ValueNorm batch moments (mb_stats / norm_rows) refer to it, so
                                    that SUM-all-reduced gradients equal the single-process gradients of the global
                                    batch; 0 = batch_rows (single process) */
} OrlPpoArgs;
/* floats per partial row for given shapes (>= folded gradient size + 8 loss slots, multiple of 4) */
int orl_ppo_stride(int obs_dim, int critic_obs_dim, int n_actions);   /* valid for both head kinds */
/* floats per net row of `grads` (>= parameter count of the larger net, multiple of 4) */
int orl_ppo_grads_stride(int obs_dim, int critic_obs_dim, int n_actions);
/* number of parameters of one MLP net with head width n (layout in DESIGN.md) */
int orl_net_param_count(int obs_dim, int n_out);
int orl_ppo_fwdbwd(const OrlPpoArgs* args, void* stream);
int orl_ppo_reduce(const OrlPpoArgs* args, void* stream);
int orl_ppo_apply(const OrlPpoArgs* args, void* stream);

/* Multi-GPU (one process per GPU): the SUM all-reduce of the gradient bucket between orl_ppo_reduce and orl_ppo_apply
 * (the north-star's "single allreduce on the gradient bucket per update"; the reference has no distributed update) fused
 * into the two kernels over NVLink peer memory instead of a separate collective.  Every rank owns one symmetric
 * allocation of orl_ppo_peer_bucket_bytes() bytes, zero-filled before first use, mapped into all peers (CUDA VMM /
 * torch symmetric memory); peer_buffers is a DEVICE array of `world` addresses of these allocations as seen from this
 * rank (entry `rank` = local_buffer).  orl_ppo_reduce_peer PUSHES this rank's bucket into slot [parity of epochs[net]]
 * [rank] of every rank's allocation; orl_ppo_apply_peer signals the peers, waits for their buckets (error_flag := 1 + peer
 * rank if one does not arrive within timeout_ms; the logged losses are then NaN), sums the `world` slots of its own copy
 * in rank order into `summed` and applies the optimiser step exactly as orl_ppo_apply does on the sum; it increments
 * epochs[net].  All ranks must issue the same sequence of reduce_peer / apply_peer pairs. */
#define ORL_PEER_MAX_WORLD 16
#define ORL_PEER_SMALL_MAX 16   /* doubles per orl_peer_sum_f64 call */
typedef struct OrlPeerArgs {
    const uint64_t* peer_buffers; /* device (world): addresses of every rank's symmetric bucket */
    float* local_buffer;          /* this rank's symmetric bucket */
    uint32_t* epochs;             /* device (3): completed exchanges {policy bucket, critic bucket, orl_peer_sum_f64}; start at 0 */
    int32_t* error_flag;          /* device (1): 0, or 1 + rank of a peer that timed out */
    float* summed;                /* device (2, stride): receives the all-rank sum (local scratch) */
    int32_t world, rank;
    int32_t timeout_ms;           /* bound on the wait for a peer's bucket */
    int32_t reserved;
} OrlPeerArgs;
long long orl_ppo_peer_bucket_bytes(int obs_dim, int critic_obs_dim, int n_actions, int world);
int orl_ppo_reduce_peer(const OrlPpoArgs* args, const OrlPeerArgs* peer, void* stream);
int orl_ppo_apply_peer(const OrlPpoArgs* args, const OrlPeerArgs* peer, void* stream);
/* In-place SUM over all ranks of n <= ORL_PEER_SMALL_MAX doubles (the 8 rollout moments of orl_gae, all-reduced once per
 * iteration: parallel.py step 1) through the same symmetric allocation; `stride` = orl_ppo_stride() of the bucket. */
int orl_peer_sum_f64(const OrlPeerArgs* peer, int stride, double* data, int n, void* stream);
/* {sum returns, sum returns^2, sum active} over a minibatch given by `indices` (see mb_stats). */
int orl_minibatch_stats(const int64_t* indices, int64_t batch_rows, const float* returns,
                        const float* active_masks, double* mb_stats_out, void* stream);


/* ---- recurrent (GRU) policy / value networks --------------------------------------------
 * Replace, for cfg.use_recurrent_policy, RNNLayer (openrl/modules/networks/utils/rnn.py:5-99) inside
 * PolicyNetwork / ValueNetwork, the recurrent half of OnPolicyDriver.act / add2buffer
 * (onpolicy_driver.py:80-152,236-279), ReplayData.recurrent_generator (replay_data.py:1062-1258:
 * chunks of L = data_chunk_length over the agent-major / time-minor flattening f = (n*A + a)*T + t,
 * initial hidden state rnn_states[f = c*L], chunks ignore trajectory boundaries) and the BPTT part of
 * PPOAlgorithm.ppo_update.  First, correctness-first implementation: one thread per row (rollout,
 * critic) or per chunk (update) running the sequential core of csrc/orl_rnn_core.h (verified on the
 * CPU against the oracle); parameter gradients are reductions of a per-row tape, dW = sum P^T Q.
 * Parameter layout of a recurrent net (reference state_dict order):
 *   W1[64][d] b1 g1 be1 | W3[64][64] b3 g3 be3 | Wih[192][64] Whh[192][64] bih bhh | g_rnn be_rnn | Wh[n][64] bh[n]
 *
 * JRPO (flags & ORL_PPO_JOINT_ACTION, cfg.use_joint_action_loss; ReplayData.recurrent_generator_v3
 * replay_data.py:425-551, _cast_v3 / _flatten_v3 buffers/utils/util.py:92-101, PPOAlgorithm.prepare_loss
 * ppo.py:222-224,254-321, ACTLayer.evaluate_actions act.py:114-118):
 *   - chunks are per env: the flattening is g = n*T + t, every g carrying all A agents; chunk c covers
 *     g in [c*L, c*L + L) (ignoring trajectory boundaries) and `chunk_ids` index these N*T / L chunks;
 *   - policy: A sequences per chunk, agent a starting from rnn_states[t0][n0*A + a] (g0 = c*L = n0*T + t0);
 *     per (chunk, step) the ratio is exp(sum_a logp_a - sum_a old_logp_a) (dual clip applies to it), the advantage
 *     and, with ORL_PPO_POLICY_ACTIVE_MASKS, the row weight are agent 0's; every agent row of the step receives
 *     the same dL/dlogp; the entropy is the mean over all agent rows (weighted by every agent's active mask with
 *     ORL_PPO_POLICY_ACTIVE_MASKS);
 *   - critic: agent 0 only (`to_single_np`): one sequence per chunk over rows n*A, n_chunks*L row-steps;
 *   - mb_stats points to 4 doubles {sum ret_0, sum ret_0^2, sum active_0, sum active_all} over the minibatch
 *     (agent 0's returns feed ValueNorm, ppo.py:190-191), norm_rows counts joint rows (chunk steps), the reported
 *     ratio is the mean joint ratio;
 *   - the tape holds n_chunks*L*A policy rows: size it with orl_rnn_workspace_floats(n_chunks*L*A, ...).
 */
typedef struct OrlRnnArgs {
    int32_t env_kind, n_envs, n_agents, episode_length;   /* N, A, T; rows B = N*A */
    int32_t t_begin, t_end;
    int32_t obs_dim, critic_obs_dim, n_actions, activation_id;
    int32_t deterministic, chunk_length;                  /* L = cfg.data_chunk_length (<= 32) */
    int32_t flags;                                        /* ORL_PPO_* */
    int32_t env_table_len;
    int64_t n_chunks;                                     /* chunks in this minibatch */
    const int64_t* chunk_ids;                             /* (n_chunks) chunk indices c (torch.randperm slice) */
    float* policy_params; float* critic_params;
    float* policy_obs; float* critic_obs;                 /* (T+1, B, d) / (T+1, B, dc) */
    float* rnn_states; float* rnn_states_critic;          /* (T+1, B, 64) */
    float* actions; float* action_log_probs; float* rewards;
    float* masks; float* active_masks;
    float* value_preds; const float* returns; const float* advantages;
    const float* exp_noise;                               /* (T, B, n) or NULL */
    uint64_t rng_seed; uint64_t rng_step_base; uint64_t* rng_counter;
    double* env_f64; uint64_t* env_u64; int32_t* env_i32; const int32_t* env_table;
    float* ep_return; int32_t* ep_length; double* episode_stats;
    const double* gae_stats; const double* mb_stats; float* vn_state;   /* mb_stats: 3 doubles (4 with ORL_PPO_JOINT_ACTION) */
    float* tape;                                          /* workspace: orl_rnn_workspace_floats(n_chunks*L, grads_stride) floats (tape rows, then reduction partials) */
    float* grads;                                         /* (2, grads_stride) true gradients, policy then critic */
    int32_t grads_stride; int32_t reserved1;
    float* loss_acc;                                      /* (8) zeroed by orl_rnn_fwdbwd: policy_loss, entropy, ratio, value_loss sums */
    float* policy_adam_m; float* policy_adam_v; float* critic_adam_m; float* critic_adam_v;
    int32_t* adam_steps; const float* lrs;
    float clip_param, entropy_coef, value_loss_coef, huber_delta, max_grad_norm;
    float adam_beta1, adam_beta2, adam_eps, weight_decay, dual_clip_coeff;
    double vn_beta;
    float* train_info;
    int64_t norm_rows;                                    /* row-steps of the GLOBAL minibatch (see OrlPpoArgs.norm_rows); 0 = n_chunks*L */
} OrlRnnArgs;
int orl_rnn_param_count(int obs_dim, int n_out);
int orl_rnn_tape_width(void);
/* floats of OrlRnnArgs.tape for a minibatch of `rows` = n_chunks * chunk_length row-steps (times n_agents with
   ORL_PPO_JOINT_ACTION) */
long long orl_rnn_workspace_floats(long long rows, int grads_stride);
/* policy GRU rollout for steps [t_begin, t_end) fused with the device env (simple_spread, CartPole, GridWorld) */
int orl_rnn_rollout(const OrlRnnArgs* args, void* stream);
/* recurrent critic over slots 0..T: value_preds[t] and rnn_states_critic[t+1] */
int orl_rnn_critic(const OrlRnnArgs* args, void* stream);
/* chunked BPTT forward + loss + backward of both nets over the minibatch chunks -> grads, loss_acc */
int orl_rnn_fwdbwd(const OrlRnnArgs* args, void* stream);
/* per-net global-norm clip + Adam on `grads`; ValueNorm commit; train_info accumulation */
int orl_rnn_apply(const OrlRnnArgs* args, void* stream);


/* ---- self-play: two-player GridWorld against an opponent pool in HBM -----------------------
 * Replaces, for BASELINE configs[3], the self-play control flow of the reference around the rollout:
 * OpponentPoolWrapper.reset / get_opponent_action / on_episode_end (openrl/selfplay/wrappers/opponent_pool_wrapper.py:
 * 30-120), RandomOpponent / LastOpponent.sample_opponent (selfplay/sample_strategy/random_opponent.py:25-28,
 * last_opponent.py:24-27); the snapshot cadence of SelfplayCallback._on_step (selfplay/callbacks/selfplay_callback.py:
 * 124-144) is the host's job (it copies the learner's parameters into the pool ring and bumps *pool_count).
 * The env (rules in csrc/orl_selfplay.cu and oracle/selfplay.py; new env, SURVEY.md §8f-2): the learner is player 0 of a
 * 10x10 two-player GridWorld and sees (x0, y0, x1, y1); player 1 is driven by the snapshot pool_params[opponent index]
 * (same policy architecture, d = 4, n = 5) drawn per episode, or acts uniformly at random while the pool is empty.
 * rollout.env_kind = ORL_ENV_GRIDWORLD_2P, rollout.env_i32 = [8][N] (x0, y0, x1, y1, steps, #resets, opponent, -),
 * rollout.env_table = optional [N][len][4] start cells, rollout.deterministic bits: 1 = greedy learner, 2 = learner
 * actions scripted from exp_noise[(t*N+e)*2 + 0], 4 = opponent actions scripted from exp_noise[(t*N+e)*2 + 1]. */
#define ORL_ENV_GRIDWORLD_2P 4
#define ORL_SP_RANDOM 0   /* RandomOpponent: uniform over the snapshots in the ring */
#define ORL_SP_LAST 1     /* LastOpponent: the newest snapshot */
typedef struct OrlSelfPlayArgs {
    OrlRolloutArgs rollout;
    const float* pool_params;    /* (pool_capacity, pool_stride) policy snapshots, flat parameter layout */
    const int32_t* pool_count;   /* (1) device: number of snapshots ever added; ring slot of snapshot k = k % pool_capacity */
    int32_t* pool_stats;         /* (pool_capacity + 1, 3) += wins / losses / draws of the training agent against each ring
                                    slot (last row: the random-action opponent), opponent_pool_wrapper.py:91-120 */
    int32_t pool_capacity, pool_stride, strategy, reserved;
} OrlSelfPlayArgs;
int orl_selfplay_reset(const OrlSelfPlayArgs* args, float* policy_obs_out, void* stream);
int orl_selfplay_rollout(const OrlSelfPlayArgs* args, void* stream);

/* ---- shared policy-value network (cfg.use_share_model) -----------------------------------
 * Replace, for cfg.use_share_model, PolicyValueNetwork (openrl/modules/networks/policy_value_network.py:33-174:
 * obs_prep MLPBase -> common MLPLayer(64, 64, layer_N=0) -> {v_out, act}) in the rollout (get_actions), the value pass
 * (get_values) and PPOAlgorithm.ppo_update with `_use_share_model` (ppo.py:46-176: both losses into one set of
 * gradients, clip_grad_norm_ over all parameters twice, ONE Adam step with lr = cfg.lr).
 * Parameter layout (named_parameters order of the reference):
 *   W1[64][d] b1 g1 be1 | W3[64][64] b3 g3 be3 | W5[64][64] b5 g5 be5 | W7[64][64] b7 g7 be7 | Wv[1][64] bv | Wa[n][64] ba
 * Discrete heads, single-agent device envs (or ORL_ENV_NONE).  OrlRolloutArgs.policy_params = the shared model.
 * OrlPpoArgs for the shared model: policy_params / policy_adam_* / lrs[0] / adam_steps[0] = the shared model and its
 * optimiser, partials = workspace of orl_share_workspace_floats() floats, grads = true gradients (>= parameter count),
 * folded = 8 floats of loss sums; critic_* fields are ignored.  With > 1 GPU the caller SUM-all-reduces `grads` and
 * `folded[0..3]` between orl_share_fwdbwd and orl_share_apply. */
int orl_share_param_count(int obs_dim, int n_actions);
int orl_share_tape_width(void);
long long orl_share_workspace_floats(long long rows, int obs_dim, int n_actions);
int orl_share_rollout(const OrlRolloutArgs* args, void* stream);
int orl_share_values(const float* params, int obs_dim, int n_actions, int activation_id, const float* obs, float* values,
                     long long rows, void* stream);
int orl_share_fwdbwd(const OrlPpoArgs* args, void* stream);
int orl_share_apply(const OrlPpoArgs* args, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OPENRL_B200_H */

/*
 * le_b200.h — C ABI of the B200-native hot path of automl/learning_environments.
 *
 * The reference is pure Python and has NO FFI layer for this path (SURVEY.md §8b): the path sits behind
 * duck-typed classes.  Each entry point below names the reference interface (file:line under
 * /root/reference) whose work it replaces; the Python mirror in learning_environments_b200/ keeps the
 * reference's class/method names and calls these through ctypes (INTEGRATION.md shows the binding).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; all `*_dev` pointers are CUDA device pointers owned by the
 *     caller (torch tensors on the host side).  `*_host` entry points take HOST pointers and do their own
 *     H2D/D2H copies (the reference-facing "plugin" call used for the end-to-end measurement).
 *   - every function returns 0 on success or a negative LE_E* code; le_last_error() gives the message
 *     (thread local).  Nothing throws or aborts across the boundary.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).  Calls are asynchronous
 *     with respect to that stream unless the name ends in _host.
 *   - Networks use the reference's torch layout: nn.Linear weight [out,in] row-major then bias
 *     (models/model_utils.py:4-39).  See "parameter vectors" below.
 */
#ifndef LE_B200_H
#define LE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LE_VERSION 100

/* error codes */
#define LE_OK 0
#define LE_EINVAL (-1)      /* bad argument / unsupported shape */
#define LE_ECUDA (-2)       /* CUDA runtime error */
#define LE_EUNSUPPORTED (-3) /* configuration outside the compiled kernel set */

/* activation ids (models/model_utils.py:9-20) */
#define LE_ACT_TANH 0
#define LE_ACT_RELU 1
#define LE_ACT_LEAKYRELU 2 /* slope 0.01 (nn.LeakyReLU default) */
#define LE_ACT_PRELU 3     /* single shared slope, init 0.25, never perturbed by NES */
#define LE_ACT_IDENTITY 4

/* training-environment kinds */
#define LE_ENV_SE 0   /* envs/virtual_env.py VirtualEnv                       */
#define LE_ENV_RN 1   /* envs/reward_env.py RewardEnv over the real env       */
#define LE_ENV_REAL 2 /* the gym env itself (envs/env_wrapper.py:51-70)       */

/* Q-network kinds */
#define LE_Q_DQN 0
#define LE_Q_DUELING 1

/* real environments (gym 0.17.3 classic_control, restated: SURVEY.md Appendix A) */
#define LE_REAL_CARTPOLE 0
#define LE_REAL_ACROBOT 1

/*
 * Parameter vectors ("theta"), float32, concatenated in state_dict order:
 *   SE  (LE_ENV_SE):  for net in (state_net[out=sd], reward_net[out=1], done_net[out=1]):
 *                        W1[H][sd+ad], b1[H], W2[out][H], b2[out]          input = cat(one_hot(a), s)
 *                     P_se = 3*H*(sd+ad+1) + H*(sd+2) + sd+2               (CartPole 2247, Acrobot 6354)
 *   RN  (LE_ENV_RN):  reward_net: W1[H][sd], b1[H], W2[1][H], b2[1]        P_rn = H*(sd+2)+1  (385)
 *   Q   (Critic_DQN): W1[H][sd], b1[H], W2[ad][H], b2[ad]                  P_q  = H*(sd+ad+1)+ad (401)
 *       general form (q_layers = L >= 1): Linear(sd,H), [Linear(H,H)] x (L-1), Linear(H,ad), each W[out][in] then b[out]
 *   Q   (Critic_DuelingDQN): feature_stream = Linear(sd,H), [Linear(H,H)] x (L-1), Linear(H,fd) (no activation after
 *       the last); value_stream = Linear(fd,fd), Linear(fd,1); advantage_stream = Linear(fd,fd), Linear(fd,ad);
 *       q = V + (A - mean over the whole batch of A)                       (CartPole yaml: 11 528 parameters)
 * PReLU slopes are not part of theta (never perturbed/updated: agents/GTN_worker.py:156-163 touches
 * nn.Linear only); they travel in le_lane_cfg.env_slope.
 */

/* One lane = one (agent, training env) pair = what ONE reference worker process runs in calc_score
 * (agents/GTN_worker.py:187-221): agents/base_agent.py:64-153 train() [+ per-episode test()] and the final
 * agents/base_agent.py:155-227 test(). */
typedef struct le_lane_cfg {
    int32_t sd, ad;         /* state / action dims (4,2 CartPole; 6,3 Acrobot)                         */
    int32_t env_kind;       /* LE_ENV_*                                                                */
    int32_t real_env;       /* LE_REAL_*: reset distribution, RN/REAL dynamics, test env               */
    int32_t env_hidden;     /* hidden width of the SE nets / the RN net (hidden_layer <= 1)            */
    int32_t env_act;        /* LE_ACT_* of the SE / RN nets                                            */
    float env_slope[3];     /* leaky/prelu slope per net (state,reward,done) or [0] for the RN         */
    int32_t rn_type;        /* reward_env_type 0,1,2,5,6 (envs/reward_env.py:84-110)                   */
    int32_t q_hidden;       /* hidden width of the Q-net / dueling feature stream (see q_layers)       */
    int32_t q_act;          /* LE_ACT_TANH | RELU | LEAKYRELU                                          */
    int32_t batch_size;     /* agents/DDQN.py:24                                                       */
    int32_t rb_size;        /* replay ring capacity (utils.py:10)                                      */
    int32_t train_episodes, test_episodes, init_episodes; /* agents/base_agent.py:16-18               */
    int32_t max_steps;      /* env._max_episode_steps (envs/env_factory.py:89)                        */
    int32_t early_out_num;  /* agents/base_agent.py:22                                                 */
    int32_t use_test_env;   /* train(env, test_env=real_env): per-episode test() feeds the reward meter */
    int32_t final_test;     /* run agent.test(real_env) after training (calc_score)                    */
    int64_t step_budget;    /* cap on training env steps: deterministic stand-in for time_remaining    */
    double gamma, lr, tau, eps_init, eps_min, eps_decay; /* agents/DDQN.py:24-32                       */
    double early_out_virtual_diff, solved_reward;        /* agents/base_agent.py:23, env config        */
    double beta1, beta2, adam_eps;                       /* torch.optim.Adam defaults .9/.999/1e-8     */
    int32_t q_kind;         /* LE_Q_DQN (models/actor_critic.py:84-91) | LE_Q_DUELING (:94-122)                */
    int32_t q_layers;       /* hidden_layer of the Q-net / feature stream (0 and 1 build the same net)         */
    int32_t q_feature_dim;  /* Critic_DuelingDQN feature_dim (heads: fd -> fd -> {1, ad})                      */
    int32_t same_action_num; /* agent same_action_num (envs/env_wrapper.py:24-61, agents/base_agent.py:104,123); 0 == 1 */
} le_lane_cfg;

/* Per-lane results (what train()/test() return, as arrays). */
typedef struct le_lane_out {
    int32_t n_episodes;     /* len(reward_list) before timeout padding                                 */
    int32_t timed_out;      /* step_budget hit (time_is_up analog, agents/base_agent.py:30-47)         */
    int64_t train_steps;    /* agent steps taken in training (each = same_action_num env steps)        */
    int64_t learn_iters;    /* DDQN.learn calls (self.it)                                              */
    int64_t test_steps;     /* real-env steps taken inside test() calls                                */
    double score;           /* statistics.mean(final test rewards) (agents/GTN_worker.py:209)          */
} le_lane_out;

/* Optional per-step trace of the first `cap` training steps of a lane (parity tests). */
typedef struct le_trace {
    int32_t cap;            /* capacity in steps; 0 disables                                           */
    int32_t* action;        /* [cap]                                                                   */
    int32_t* explore;       /* [cap] 1 if the action was random                                        */
    float* next_state;      /* [cap*sd]                                                                */
    float* reward;          /* [cap]                                                                   */
    float* done;            /* [cap]                                                                   */
    float* loss;            /* [cap] NaN when no learn() happened on that step                         */
    float* qgap;            /* NULL or [cap]: greedy steps: (q_best - q_second) / max(|q_best|, |q_second|, 1e-12) of the
                               Q-values the action was chosen from (a near-tie marker for the parity tests); NaN when the
                               action was random                                                         */
} le_trace;

/* ------------------------------------------------------------------------------------------------ */
/* library                                                                                          */
int le_version(void);
const char* le_last_error(void);
int le_sizeof_lane_cfg(void); /* ABI check for bindings */
/* number of SMs / name of the current device (diagnostics for bench.py) */
int le_device_info(int device, int* sm_count, int* cc_major, int* cc_minor, char* name, int name_cap);

/* Measured FP32 FFMA throughput of the current device in TFLOP/s (microbenchmark; the roofline denominator
 * of the FFMA-bound fused kernel — MEASURED_PEAKS.json carries only HBM and bf16-tensor peaks). */
int le_bench_ffma(int iters, int reps, double* tflops_out, void* stream);

/* ------------------------------------------------------------------------------------------------ */
/* unit operators (one reference call each), batched over `n` independent rows/lanes                 */

/* VirtualEnv.step (envs/virtual_env.py:43-54) through EnvWrapper.step (envs/env_wrapper.py:17-49):
 * n = pop*lanes rows; row r uses theta of member r / lanes_per_member.                               */
int le_se_forward(const le_lane_cfg* cfg, const float* theta_dev /*[pop][P_se]*/, int pop, int lanes_per_member,
                  const float* state_dev /*[n][sd]*/, const int32_t* action_dev /*[n]*/,
                  float* next_state_dev /*[n][sd]*/, float* reward_dev /*[n]*/, float* done_dev /*[n]*/,
                  void* stream);

/* RewardEnv._calc_reward (envs/reward_env.py:68-133) for types 0,1,2,5,6: n rows, one theta per member. */
int le_rn_reward(const le_lane_cfg* cfg, const float* theta_dev /*[pop][P_rn]*/, int pop, int lanes_per_member,
                 const float* state_dev, const float* next_state_dev, const float* real_reward_dev,
                 float* reward_dev, void* stream);

/* Critic_DQN.forward / Critic_DuelingDQN.forward (models/actor_critic.py:84-122) + greedy argmax
 * (agents/DDQN.py:106-110): one Q-net per lane (q_theta [n][P_q]), one state row per lane.            */
int le_qnet_forward(const le_lane_cfg* cfg, const float* q_theta_dev, int n, const float* state_dev,
                    float* q_out_dev /*[n][ad]*/, int32_t* argmax_dev /*[n]*/, void* stream);

/* gym CartPole/Acrobot step + TimeLimit (SURVEY Appendix A; envs/env_wrapper.py:51-70): fp64 state in/out. */
int le_real_env_step(int real_env, int max_steps, double* state_dev /*[n][4]*/, int32_t* elapsed_dev /*[n]*/,
                     const int32_t* action_dev, float* obs_dev /*[n][sd]*/, float* reward_dev, float* done_dev,
                     int n, void* stream);

/* DDQN.learn (agents/DDQN.py:60-95) / DuelingDDQN.learn (agents/DuelingDDQN.py:59-94) on explicit minibatches:
 * per lane B rows [s(sd) a s'(sd) r d] packed
 * (2*sd+3 floats).  Updates q_theta/q_target/m/v in place, t_dev[n] is Adam's step count, loss_dev[n] out. */
int le_td_update(const le_lane_cfg* cfg, float* q_theta_dev, float* q_target_dev, float* adam_m_dev,
                 float* adam_v_dev, int32_t* adam_t_dev, int n, const float* batch_rows_dev /*[n][B][2sd+3]*/,
                 float* loss_dev, void* stream);

/* One dense-layer GEMM on the tcgen05 tensor cores (3xTF32, fp32 accumulate in TMEM) with the contract of the general
 * kernel's dense layers: C[i*c_si + j*c_sj] (+)= sum_l A[i*a_si + l*a_sl] * B[l*b_sl + j*b_sj] (+ bias[j], activation
 * act: 0 identity, 1 tanh, 2 leaky family with `slope`).  Covers nn.Linear forward (models/model_utils.py:22-36, X W^T),
 * its input gradient (dZ W) and weight gradient (dZ^T X) as torch.autograd computes them for DDQN.learn /
 * DuelingDDQN.learn (agents/DuelingDDQN.py:59-94).  Unit operator for the parity tests; the lane kernels call the same
 * device routine (csrc/le_tc.cuh). */
int le_tc_gemm(const float* A_dev, int a_si, int a_sl, const float* B_dev, int b_sl, int b_sj, float* C_dev, int c_si, int c_sj,
               int I, int J, int L, const float* bias_dev, int act, float slope, int accumulate, void* stream);

/* ------------------------------------------------------------------------------------------------ */
/* the fused hot path                                                                               */

/* Bytes of device workspace needed for n lanes sharing n_env environment parameter vectors: the packed
 * SE/RN weights, one replay ring per RESIDENT warp slot (not per lane) and the lane queue counter.
 * Returns a negative LE_E* code on error. */
int64_t le_inner_loop_workspace_bytes(const le_lane_cfg* cfg, int n_lanes, int n_env);

/* The launch plan behind the two calls above/below (diagnostics for bench.py / DESIGN.md): CTAs, resident
 * warp slots, replay ring capacity in rows, hidden units per thread of the selected kernel set. */
int le_inner_loop_plan(const le_lane_cfg* cfg, int n_lanes, int n_env, int* grid, int* slots, int* ring_cap, int* units,
                       int64_t* ring_offset_bytes /* offset of warp slot 0's replay ring inside the workspace */);

/*
 * Runs n_lanes complete `calc_score`s (agents/GTN_worker.py:187-221) — train() with ε-greedy acting
 * (agents/DDQN.py:97-104), SE/RN/real env step, replay append (utils.py:24-32), TD update
 * (agents/DDQN.py:60-95), per-episode greedy test() on the real env, early-out (agents/base_agent.py:49-62)
 * and the final test() — in ONE persistent kernel: one warp per lane for Critic_DQN with hidden_layer <= 1 and
 * hidden_size <= 128 (weights in registers), one 256-thread CTA per lane for every other Q-net (DuelingDDQN,
 * two hidden layers, wider nets).  Lanes of one launch must all fall into the same of the two families.
 *
 *   cfg_dev        [n_cfg] lane configurations (DEVICE); lane i uses cfg_dev[n_cfg == 1 ? 0 : i]  (vary_hp:
 *                  per-lane lr / batch_size / q_hidden <= cfg_host0->q_hidden).  cfg_host0 = HOST copy of the
 *                  configuration that fixes shapes, strides and the ring capacity (cfg 0 / the maxima)
 *   env_theta_dev  [n_env][P_env]; lane i uses row env_index_dev[i] (NULL: row 0)
 *   keys_dev       [n_lanes][2] Philox lane keys
 *   q_init_dev     NULL: Q-nets are initialised on device from the P_QINIT stream (torch default init
 *                  distribution, models/model_utils.py:31); else [n_lanes][P_q] initial weights
 *   q_final_dev    NULL or [n_lanes][P_q]: trained online-net weights out
 *   out_dev        [n_lanes] le_lane_out
 *   rewards_dev    [n_lanes][train_episodes] doubles: avg_meter_reward raw data (base_agent.py:153)
 *   lengths_dev    [n_lanes][train_episodes] int32: episode lengths
 *   test_rewards_dev [n_lanes][test_episodes] doubles: final test() rewards
 *   test_lengths_dev NULL or [n_lanes][test_episodes] int32: final test() episode lengths
 *   workspace_dev  le_inner_loop_workspace_bytes() bytes
 *   trace_dev      NULL or one le_trace (device pointers inside) that records lane `trace_lane`
 */
int le_inner_loop_run(const le_lane_cfg* cfg_dev, int n_cfg, const le_lane_cfg* cfg_host0,
                      const float* env_theta_dev, int n_env, const int32_t* env_index_dev, const uint32_t* keys_dev,
                      const float* q_init_dev, float* q_final_dev, int n_lanes, le_lane_out* out_dev,
                      double* rewards_dev, int32_t* lengths_dev, double* test_rewards_dev, int32_t* test_lengths_dev,
                      void* workspace_dev, int64_t workspace_bytes, const le_trace* trace_host, int trace_lane, void* stream);

/* Host-buffer convenience wrapper of le_inner_loop_run (the reference-facing call a GTN worker would
 * make: everything in host memory, H2D/D2H inside).  Arrays as above but HOST pointers.              */
int le_inner_loop_run_host(const le_lane_cfg* cfgs, int n_cfg, const float* env_theta, int n_env,
                           const int32_t* env_index, const uint32_t* keys, const float* q_init, float* q_final,
                           int n_lanes, le_lane_out* out, double* rewards, int32_t* lengths,
                           double* test_rewards, int device);

/* ------------------------------------------------------------------------------------------------ */
/* TD3_discrete_vary lanes (SURVEY.md §8(f) rank 2; agents/TD3_discrete_vary.py, models/actor_critic.py:22-36,69-76)  */

/* base: env / loop / Adam fields as for DDQN lanes (eps_* unused); q_hidden, q_layers, q_act give the shape of the actor
 * (sd -> H x L -> ad) and of the two critics (sd+ad -> H x L -> 1). */
typedef struct le_td3_cfg {
    le_lane_cfg base;
    int32_t policy_delay;    /* agents/TD3_discrete_vary.py:35 */
    int32_t gumbel_hard;     /* gumbel_softmax_hard (models/actor_critic.py:32) */
    double action_std, policy_std, policy_std_clip; /* :37-39 */
    double gumbel_temp;      /* gumbel_softmax_temp, annealed to /20 over 2000 learn() calls (:58-59) */
    double max_action;       /* envs/env_wrapper.py:106-110 */
} le_td3_cfg;

/* n_lanes complete train(+per-episode test)+test runs of TD3_discrete_vary agents (the DDQN lanes' le_inner_loop_run_host
 * for this agent family), HOST buffers in and out.  actor_init [n_init][P_actor], critic1_init / critic2_init
 * [n_init][P_critic] with n_init = 1 (shared by all lanes) or n_lanes; parameter vectors in torch state_dict order.
 * Training env: LE_ENV_SE or LE_ENV_REAL.  trace_host (may be NULL): HOST arrays recording lane `trace_lane`.           */
int le_td3_param_counts(const le_td3_cfg* cfg, int* p_actor, int* p_critic);

/* Bytes of device workspace for le_td3_run: the packed SE weights, the lane queue counter and one slot (replay ring, the six
 * nets, Adam state, minibatch activations) per RESIDENT lane, every slot sized for cfg_host0 (the maxima of the launch).
 * When the slots of all resident lanes do not fit 90 % of the free device memory, the size asks for fewer slots (at least
 * one); le_td3_run then keeps fewer lanes resident and queues the rest.  Returns a negative LE_E* code on error. */
int64_t le_td3_workspace_bytes(const le_td3_cfg* cfg_host0, int n_lanes, int n_env);

/*
 * The TD3 counterpart of le_inner_loop_run: n_lanes TD3_discrete_vary agents, one 256-thread CTA per lane, DEVICE buffers,
 * asynchronous on `stream`.  vary_hp batches of transfer evaluations run here in one launch.
 *   cfg_dev        [n_cfg] configurations (DEVICE); lane i uses cfg_dev[n_cfg == 1 ? 0 : i] with its own q_hidden, q_layers,
 *                  batch_size, lr, ...; cfg_host0 = HOST copy of the maxima (q_hidden, q_layers, batch_size) that sizes the
 *                  slots, and the configuration whose env / loop fields fix the ring capacity and the result strides
 *   env_theta_dev  [n_env][P_se]; lane i uses row env_index_dev[i] (NULL: row 0); NULL for LE_ENV_REAL
 *   keys_dev       [n_lanes][2] Philox lane keys
 *   actor_init_dev / critic1_init_dev / critic2_init_dev   all NULL: every lane initialises its three nets on the device
 *                  (torch default nn.Linear init from the P_TD3_INIT stream, restated in tests/td3_init_stream.py); else [n_init][P] with
 *                  n_init = 1 (shared) or n_lanes, row stride = the parameter counts of cfg_host0 (le_td3_param_counts)
 *   actor_final_dev NULL or [n_lanes][P_actor of cfg_host0]: trained actors (the first P_actor of lane i's own shape)
 *   out_dev, rewards_dev, lengths_dev, test_rewards_dev   as for le_inner_loop_run
 *   workspace_dev  le_td3_workspace_bytes() bytes (a smaller workspace that holds at least one slot runs fewer lanes at once)
 *   trace_host     NULL or one le_trace (DEVICE pointers inside) that records lane `trace_lane`
 * Training env: LE_ENV_SE or LE_ENV_REAL (LE_ENV_RN: LE_EUNSUPPORTED).
 */
int le_td3_run(const le_td3_cfg* cfg_dev, int n_cfg, const le_td3_cfg* cfg_host0, const float* env_theta_dev, int n_env,
               const int32_t* env_index_dev, const uint32_t* keys_dev, const float* actor_init_dev, const float* critic1_init_dev,
               const float* critic2_init_dev, int n_init, float* actor_final_dev, int n_lanes, le_lane_out* out_dev, double* rewards_dev,
               int32_t* lengths_dev, double* test_rewards_dev, void* workspace_dev, int64_t workspace_bytes, const le_trace* trace_host,
               int trace_lane, void* stream);

/* Host-buffer wrapper of le_td3_run with one configuration for all lanes (arrays as above, HOST pointers). */
int le_td3_run_host(const le_td3_cfg* cfg, const float* env_theta, int n_env, const int32_t* env_index, const uint32_t* keys,
                    const float* actor_init, const float* critic1_init, const float* critic2_init, int n_init, float* actor_final,
                    int n_lanes, le_lane_out* out, double* rewards, int32_t* lengths, double* test_rewards,
                    const le_trace* trace_host, int trace_lane, int device);

/* ------------------------------------------------------------------------------------------------ */
/* NES outer step (agents/GTN_worker.py:156-185, agents/GTN_master.py:267-298)                        */

/* get_random_noise + add_noise (+/-): out[(m*3+v)][P] = theta + sign_v * noise_std * N(0,1), v in
 * {0: theta, 1: +eps, 2: -eps}; normals from Philox (seed, generation, member) — never stored.        */
int le_nes_perturb(const float* theta_dev /*[P]*/, int P, int pop, int member_offset, int n_members,
                   uint32_t seed, uint32_t generation, float noise_std, float* out_dev /*[n_members*3][P]*/,
                   void* stream);

/* The raw noise eps_i = noise_std * N(0,1) for members [member_offset, member_offset+n) (debug/tests). */
int le_nes_noise(int P, int member_offset, int n_members, uint32_t seed, uint32_t generation, float noise_std,
                 float* eps_dev /*[n_members][P]*/, void* stream);

/* update_env: theta <- theta*(1-wd); for i in 0..pop-1 (in order): theta += coef[i]*sign[i]*eps_i, with
 * eps_i regenerated from Philox; coef[i] = (float)(step_size * score_transform[i]).                   */
int le_nes_update(float* theta_dev /*[P]*/, int P, int pop, uint32_t seed, uint32_t generation,
                  float noise_std, double weight_decay, const float* coef_dev /*[pop]*/,
                  const float* sign_dev /*[pop] +1/-1*/, void* stream);

/* Partial (sharded) form for the allreduce path: delta[P] = sum_{i in [lo,hi)} coef[i]*sign[i]*eps_i.    */
int le_nes_partial_update(float* delta_dev /*[P]*/, int P, int member_lo, int member_hi, uint32_t seed,
                          uint32_t generation, float noise_std, const float* coef_dev, const float* sign_dev,
                          void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LE_B200_H */

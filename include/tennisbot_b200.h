/* tennisbot_b200.h - C ABI of the B200 env-step library (libtennisbot_b200.so).
 *
 * The reference has no FFI of its own: its two gym envs call the `pybullet` CPython extension directly.  This
 * header is the boundary a maintainer binds instead (ctypes stub in INTEGRATION.md); each entry point names the
 * reference code it replaces (paths relative to the reference checkout).
 *
 * Conventions
 *  - opaque context per (device, env kind, batch size); one context = one lock-step batch of N envs whose
 *    state lives in HBM, structure-of-arrays, owned by the library;
 *  - every `d_*` argument is a caller-owned DEVICE pointer (e.g. a torch tensor's data_ptr()), `h_*` is a HOST
 *    pointer; `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *  - calls on one context are stream-ordered and not re-entrant; distinct contexts are independent;
 *  - every function returns 0 on success, non-zero on failure with a thread-local message in tb_last_error();
 *    no C++ exception, Python object or torch type crosses the boundary;
 *  - there is no CPU fallback: tb_create fails when no sm_100 device is usable.
 */
#ifndef TENNISBOT_B200_H
#define TENNISBOT_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TB_ABI_VERSION 1

/* env kinds: gym ids registered in tennisbot/__init__.py:3-11 */
#define TB_ENV_SWING 0 /* "SwingRacket-v0" -> tennisbot/envs/swingracket_env.py */
#define TB_ENV_HIT 1   /* "Tennisbot-v0"   -> tennisbot/envs/tennisbot_env.py   */

/* arithmetic type of the state and of every in-kernel computation */
#define TB_F32 0
#define TB_F64 1 /* what Bullet computes in (double-precision build); event-exact against the oracle */

#define TB_STATE_WORDS 32 /* canonical per-env state record of tb_get_state / tb_set_state (doubles) */
#define TB_INIT_WORDS 8   /* explicit placement record of tb_reset_from (doubles) */
#define TB_NUM_STATS 10

/* canonical state record (same layout the CPU oracle uses) */
#define TB_S_RACKET_POS 0   /* COM position = pybullet.getBasePositionAndOrientation (racket.py:131) */
#define TB_S_RACKET_QUAT 3  /* x,y,z,w */
#define TB_S_RACKET_VEL 7   /* getBaseVelocity linear (racket.py:142) */
#define TB_S_RACKET_ANGVEL 10
#define TB_S_BALL_POS 13    /* objects.py:57 */
#define TB_S_BALL_VEL 16    /* objects.py:64 */
#define TB_S_BALL_ANGVEL 19
#define TB_S_AUX 22         /* swing: spawn_pos (swingracket_env.py:166); hit: ball_shoot_force (tennisbot_env.py:237) */
#define TB_S_GOAL 25        /* swing: goal x,y (swingracket_env.py:173) */
#define TB_S_D0 27          /* swing: initial_dist_to_goal (swingracket_env.py:174) */
#define TB_S_RETURN 28
#define TB_S_STEP 29        /* step_count */
#define TB_S_FLAGS 30       /* bit0: done */
#define TB_S_EPISODE 31     /* episode index = RNG counter word */

/* per-step event bits */
#define TB_EV_RACKET_BALL 1  /* len(getContactPoints(racket, ball)) > 0  (swingracket_env.py:99, tennisbot_env.py:170) */
#define TB_EV_COURT_BALL 2   /* len(getContactPoints(court, ball)) > 0   (swingracket_env.py:111) */
#define TB_EV_GOAL_BALL 4    /* len(getContactPoints(goal, ball)) > 0    (swingracket_env.py:119) */
#define TB_EV_TIMEOUT 8      /* step_count > 800 / > 1000                (swingracket_env.py:127, tennisbot_env.py:201) */
#define TB_EV_BALL_PASSED 16 /* ball_x - racket_x >= 0.5                 (tennisbot_env.py:182-194) */
#define TB_EV_NET_BALL 32    /* the court contact was with the net box */
#define TB_EV_RACKET_LOW 64  /* racket hull reached the floor plane; racket-court contact is not modelled */

/* statistics vector (int64, exact and order independent; sums of floats are fixed point) */
#define TB_STAT_EPISODES 0
#define TB_STAT_SUM_LENGTH 1
#define TB_STAT_RACKET_HITS 2  /* rewarded racket-ball contact steps */
#define TB_STAT_GOALS 3
#define TB_STAT_COURT 4
#define TB_STAT_TIMEOUTS 5
#define TB_STAT_SUM_RETURN_Q20 6   /* sum of round(return * 2^20) */
#define TB_STAT_SUM_RETURN2_Q10 7  /* sum of round(return^2 * 2^10) */
#define TB_STAT_PHYSICS_STEPS 8
#define TB_STAT_ENV_STEPS 9

/* how an action drives the racket */
#define TB_CONTROL_FORCE 0 /* Racket.apply_target_action: world-frame force / torque at the COM (racket.py:92-100);
                              what both registered gym envs do (swingracket_env.py:76-79, tennisbot_env.py:112-115) */
#define TB_CONTROL_PID 1   /* Racket.apply_action = set_target_location + apply_pid_force_torque (racket.py:66-89,
                              103-122): action[0:3] is a target position (hit env: action[0:2] + z = pid_hit_z), three
                              simple_pid controllers evaluated in-kernel, force = (0,0,pid_bias_z) + outputs.  Reachable in
                              the reference from playground.py:70-106 and the commented call at tennisbot_env.py:107 */

/* in-kernel action sources for tb_rollout */
#define TB_ACT_RANDOM 0 /* U(-1,1) = action_space.sample(); Philox stream keyed (env, episode, step) */
#define TB_ACT_TRACK 1  /* Tennisbot-v0 only: scripted ball tracker, a0 = 0.2 U(-1,1), a1 = clip(4 (ball_y - racket_y) - 1.5
                           racket_vy, -1, 1) in float32 on the observation entries: BASELINE config 3 "with racket-ball
                           contact" (uniform actions meet the ball in ~2 % of episodes) */

typedef struct tb_ctx tb_ctx;

typedef struct tb_config {
  uint32_t struct_size;  /* sizeof(tb_config), for forward compatibility */
  int32_t env_kind;      /* TB_ENV_* */
  int32_t precision;     /* TB_F32 / TB_F64 */
  int32_t device;        /* CUDA device ordinal */
  int64_t num_envs;      /* N, envs stepped in lock step by this context */
  int64_t env_id_offset; /* global id of env 0: RNG streams are keyed by global id, so a batch sharded over
                            several GPUs reproduces the single-GPU batch */
  uint64_t seed;
  int32_t auto_reset;    /* 1: a done env starts its next episode inside the same step (VecEnv semantics);
                            0: gym.Env semantics, the caller resets (swingracket_env.py:151) */
  int32_t reserved;
} tb_config;

/* ---- introspection; callable without a GPU */
const char *tb_last_error(void);
int tb_abi_version(void);
int tb_obs_dim(int env_kind);   /* observation_space.shape[0]: 6 (swingracket_env.py:34-39) / 12 (tennisbot_env.py:51-55) */
int tb_act_dim(int env_kind);   /* action_space.shape[0]:      6 (swingracket_env.py:29-31) / 2  (tennisbot_env.py:37-44) */
int tb_policy_floats(int env_kind); /* floats tb_set_policy expects: TB_POLICY_FLOATS / TB_POLICY_FLOATS_HIT (-1: unknown kind) */
int tb_num_params(void);
const char *tb_param_name(int index);
/* scene constants as compiled into the library (masses, radii, hull outline ...), for the fixture cross-check */
int tb_scene_constant(const char *name, int index, double *value);

/* ---- lifetime.  Replaces p.connect(DIRECT) + p.resetSimulation + loadURDF x4 (swingracket_env.py:44-47,153-182) */
int tb_create(const tb_config *cfg, tb_ctx **out);
int tb_destroy(tb_ctx *ctx); /* p.disconnect (swingracket_env.py:189) */

/* every recalled Bullet constant is a named parameter (SURVEY.md Appendix A); also "racket_scale"
 * = TennisbotEnv.set_racket_scale / loadURDF(globalScaling) (tennisbot_env.py:213-215, racket.py:39) */
int tb_set_param(tb_ctx *ctx, const char *name, double value);
int tb_get_param(tb_ctx *ctx, const char *name, double *value);
/* TB_CONTROL_*; PID gains / limits are the parameters pid_kp, pid_ki, pid_kd, pid_max_force (Racket.update_pid,
 * racket.py:170-184), pid_bias_z, pid_hit_z.  Controller memory is per env and cleared by reset. */
int tb_set_control_mode(tb_ctx *ctx, int mode);

/* ---- reset(): swingracket_env.py:151-186, tennisbot_env.py:217-261.
 * Starts a new episode for envs with d_mask[i] != 0 (all if NULL).  d_obs float32 [N, obs_dim] (may be NULL). */
int tb_reset(tb_ctx *ctx, const uint8_t *d_mask, float *d_obs, void *stream);
/* same with explicit placement instead of the RNG.  d_init double [N, TB_INIT_WORDS]:
 *   swing: racket base x,y,z, goal x,y, 0,0,0 ; hit: racket base x,y,z, shoot force x,y, ball x,y,z */
int tb_reset_from(tb_ctx *ctx, const double *d_init, const uint8_t *d_mask, float *d_obs, void *stream);

/* ---- step(): swingracket_env.py:75-145, tennisbot_env.py:104-207 (+ p.stepSimulation, p.getContactPoints,
 * Racket.apply_target_action racket.py:92-100, Ball.apply_force objects.py:67-72).  Two launches on `stream`:
 * step_kernel (every env, one substep) and, for SwingRacket, ff_kernel (the queued fast-forward flights).
 * d_actions float32 [N, act_dim]; d_obs float32 [N, obs_dim]; d_reward float32 [N]; d_done uint8 [N];
 * d_terminal_obs float32 [N, obs_dim] written for done envs only (may be NULL); d_events uint8 [N] (may be NULL).
 * Never synchronises with the host and keeps all per-step bookkeeping (queue counters, slot tags) in device memory, so
 * any number of tb_step calls on a stream can be captured into a CUDA graph and replayed. */
int tb_step(tb_ctx *ctx, const float *d_actions, float *d_obs, float *d_reward, uint8_t *d_done,
            float *d_terminal_obs, uint8_t *d_events, void *stream);

/* K env steps fused in one launch with actions produced in-kernel (state stays in registers across them).
 * d_obs: observation after the last step; d_reward_sum float32 [N]; d_done_count int32 [N] (any may be NULL). */
int tb_rollout(tb_ctx *ctx, int action_mode, int k_steps, float *d_obs, float *d_reward_sum, int32_t *d_done_count,
               void *stream);

/* ---- policy rollout (SURVEY 8(f)-1): what SB3's collect_rollouts does around env.step (train_swing.py:83-122), kept on the
 * device.  The policy is the one the reference trains: SB3 MlpPolicy with net_arch pi = vf = [32, 64, 32], tanh, a Gaussian
 * head with state-independent log_std (train_swing.py:80-91; backup_models/ppo_swing.zip).  Tennisbot-v0 uses the same
 * towers on its 12 inputs and 2 outputs (train.py's net_arch is not recorded).  Parameters, float32, each tensor row-major
 * [out][in] and padded to a multiple of 4 floats.  SwingRacket-v0 (obs_dim 6, act_dim 6):
 *   pi tower: W1[32x6] b1[32] W2[64x32] b2[64] W3[32x64] b3[32] action_net W[6x32] b[6 -> 8]                (4616 floats)
 *   vf tower: W1 b1 W2 b2 W3 b3 (same shapes) value_net W[1x32] b[1 -> 4]                                   (4452 floats)
 *   log_std[6 -> 8]                                                                                          (8 floats)
 * Tennisbot-v0 (obs_dim 12, act_dim 2):
 *   pi tower: W1[32x12] b1[32] W2[64x32] b2[64] W3[32x64] b3[32] action_net W[2x32] b[2 -> 4]               (4676 floats)
 *   vf tower: W1 b1 W2 b2 W3 b3 (same shapes) value_net W[1x32] b[1 -> 4]                                   (4644 floats)
 *   log_std[2 -> 4]                                                                                          (4 floats) */
#define TB_POLICY_FLOATS 9076
#define TB_POLICY_FLOATS_HIT 9324
/* count must be tb_policy_floats(env_kind).  Returns the context to one policy after tb_set_policies. */
int tb_set_policy(tb_ctx *ctx, const float *d_params, int64_t count, void *stream);
/* A population of policies for one context: d_params float32 [agents, tb_policy_floats(env_kind)], rows in tb_set_policy's
 * layout.  agents >= 1 must divide N; env i acts with agent i / (N / agents).  Like tb_set_policy, a stream-ordered device to
 * device copy into a library-owned buffer: it never synchronises, can be captured, and a replayed graph copies the weights
 * d_params holds at replay time.  A call that needs more floats than the buffer holds allocates a larger one (cudaMalloc, and
 * cudaFree of the old one, which waits for the device): make the largest call before capturing, and capture again after a
 * call that grew the buffer, since graphs captured earlier refer to the old one.  Fails on a NULL d_params, agents < 1,
 * agents not dividing N, count != agents x tb_policy_floats(env_kind), and on a faulted context.  agents = 1 is
 * tb_set_policy. */
int tb_set_policies(tb_ctx *ctx, const float *d_params, int64_t agents, int64_t count, void *stream);
/* K env steps with actions sampled from the policy: per step one policy_kernel launch (forward, Philox Gaussian noise,
 * log-density, value) followed by tb_step's launches, all on `stream`, nothing synchronises - capturable in a CUDA graph.
 * d_obs float32 [K, N, obs_dim]: d_obs[0] must hold the current observation (from tb_reset or the previous rollout's
 * d_last_obs); d_obs[t] receives the observation step t acted on.  d_actions float32 [K, N, act_dim]: the sampled, UNCLIPPED
 * action (env.step gets it clipped to the Box, as SB3 does); d_logp, d_value float32 [K, N]; d_reward float32 [K, N];
 * d_done uint8 [K, N]; d_last_obs float32 [N, obs_dim] and d_last_value float32 [N]: observation after the last step and its
 * value (GAE bootstrap).  d_actions, d_logp, d_value, d_last_value may be NULL.  deterministic = 1: action = mean
 * (model.predict(deterministic=True)); else stochastic, as validate_swing.py:35 rolls the policy.  The noise streams
 * are keyed (noise_seed, global env id, the context's env-step counter, a device word): independent of the env's own streams
 * and of the sharding, and fresh on every replay of a captured graph.
 * After tb_set_policies with agents > 1, env i acts with agent i / (N / agents): every buffer, the noise and the launch count
 * stay as they are, so agent p's envs give what a context of N / agents envs with env_id_offset = p N / agents and the same
 * seeds gives with that agent's policy.  tb_read_stats still sums over the whole context.  With a normaliser attached, the
 * P policies and the A records of tb_set_vecnorms must agree: P = A = 1 is the one-record rollout, P = A > 1 normalises env i
 * with record i / (N / A), so agent p's envs also give what the shard gives with record p attached by tb_set_vecnorm; any
 * other pair fails, naming both counts. */
int tb_policy_rollout(tb_ctx *ctx, int k_steps, int deterministic, uint64_t noise_seed, float *d_obs, float *d_actions,
                      float *d_logp, float *d_value, float *d_reward, uint8_t *d_done, float *d_last_obs,
                      float *d_last_value, void *stream);
/* tb_policy_rollout that also returns the env's reward before normalisation: d_raw_reward float32 [K, N] (may be NULL, which is
 * tb_policy_rollout).  Each step's raw reward is copied there with one cudaMemcpyAsync device to device right after the step,
 * which is not a kernel launch: the launch count is tb_policy_rollout's.  Without a normaliser it equals d_reward.  With
 * norm_reward, d_reward comes back normalised by each agent's own record, so per-agent episode returns are summed from
 * d_raw_reward. */
int tb_policy_rollout_raw(tb_ctx *ctx, int k_steps, int deterministic, uint64_t noise_seed, float *d_obs, float *d_actions,
                          float *d_logp, float *d_value, float *d_reward, float *d_raw_reward, uint8_t *d_done,
                          float *d_last_obs, float *d_last_value, void *stream);

/* ---- observation and reward normalisation of the policy rollout: SB3 1.8 VecNormalize, on the device.
 * Statistics, float64, RunningMeanStd layout: obs mean [obs_dim], obs var [obs_dim], obs count, ret mean, ret var, ret count
 * (TB_VECNORM_WORDS doubles); fresh: means 0, variances 1, counts 1e-4 (RunningMeanStd(epsilon=1e-4)).  Per-env discounted
 * returns, float64 [N], belong to the context and are not part of the record (SB3 drops `returns` when it pickles).
 * An update with the N envs' values of a batch (population variance b_var, mean b_mean, count N) is Chan's merge, as
 * RunningMeanStd.update_from_moments: delta = b_mean - mean, tot = count + N, mean += delta N / tot,
 * var = (var count + b_var N + delta^2 count N / tot) / tot, count = tot.  The batch moments are formed in float64 from the
 * float32 values in a fixed reduction order (the ES normaliser's pairwise merges); SB3's np.mean of a float32 array sums in
 * float32, so the library deliberately differs from SB3 in that rounding.
 * With a normaliser attached, env step t of tb_policy_rollout (raw observation o_t, action, raw r_t, done_t, raw o_{t+1}):
 *   1. training && norm_obs: fold o_{t+1} of all N envs (an auto-reset env's reset observation included) into the obs stats;
 *   2. training: returns = returns * gamma + r_t, folded into the return stats;
 *   3. r^_t = clip(r_t / sqrt(ret_var + epsilon), +-clip_reward) if norm_reward, else r_t; then returns[done_t] = 0;
 *   4. o^ = clip((o - obs_mean) / sqrt(obs_var + epsilon), +-clip_obs) if norm_obs, else o: float64 with every operation
 *      rounded (no contraction), rounded once to float32, so numpy float64 on the same statistics reproduces it bit for bit.
 *      The policy acts on o^ (and the value is that of o^).
 * The first rollout after tb_set_vecnorm, or after a tb_reset / tb_reset_from of all envs (mask NULL), first folds its
 * d_obs[0] (SB3's reset() does); those calls zero the returns, a masked reset zeroes the returns of the envs it resets and
 * folds nothing.  training = 0: the statistics and returns never change (deployment).
 * tb_policy_rollout's buffers change meaning with a normaliser only: d_obs[0] holds the RAW current observation on entry;
 * on return d_obs[t] holds the normalised observation step t acted on (t = 0 included), d_reward[t] = r^_t, d_last_obs the
 * RAW observation after the last step (the next call's d_obs[0]) and d_last_value the value of its normalised form.
 * Kernel launches of tb_policy_rollout with a normaliser: K (3 + s) + 3 when training (an entry pass of 2 launches that folds
 * d_obs[0] when armed, and two statistics launches after each step), K (1 + s) + 2 when not; s = 2 for SwingRacket-v0 and 1 for
 * Tennisbot-v0 (tb_step's launches), and the last launch (bootstrap value, last normalised reward) always runs.  tb_reset /
 * tb_reset_from add one launch while a training normaliser is attached.  The int64 statistics (tb_read_stats) stay raw;
 * tb_step, tb_rollout, tb_reset_host, tb_step_host and the ES entry points ignore the normaliser, and so does tb_sac_rollout
 * unless its mode carries TB_SAC_VECNORM (see there; tb_vecnorm_apply normalises replay samples).  Each context keeps its
 * own statistics: shards with env_id_offset do not reproduce the statistics of one batch.
 * A population (tb_set_policies) normalises with one record per agent (tb_set_vecnorms): every rule above holds per agent,
 * over that agent's N / A envs, and the statistics pass stays two launches (a segmented pass: es_norm_blocks(N / A) CTAs per
 * agent, laid out as a context of N / A envs lays them out, then one CTA per agent), so record p is bit for bit the record of a
 * context of N / A envs at env_id_offset p N / A.  The launch counts above hold for any A.  One armed byte serves the context:
 * a full reset resets every agent. */
typedef struct tb_vecnorm {
  uint32_t struct_size; /* sizeof(tb_vecnorm) */
  int32_t training, norm_obs, norm_reward;
  double clip_obs, clip_reward, gamma, epsilon; /* SB3's defaults: 10, 10, 0.99, 1e-8 */
} tb_vecnorm;
#define TB_VECNORM_WORDS(obs_dim) (2 * (obs_dim) + 4) /* obs mean, obs var, obs count, ret mean, ret var, ret count */
/* Attach (cfg) or detach (cfg NULL) the normaliser.  d_stats double [TB_VECNORM_WORDS(obs_dim)]: the record to start from (NULL:
 * fresh); the call copies it to the host and checks it, so with d_stats it synchronises `stream`; otherwise it is one kernel
 * launch and never synchronises.  Zeroes the returns and arms the reset fold.  Fails on a wrong struct_size, clip_obs or
 * clip_reward or epsilon that is not finite and above 0, gamma outside [0, 1], stats with a count <= 0, a variance < 0 or an
 * entry that is not finite, and on a faulted context.  Detaching keeps the buffers; attaching again starts from d_stats. */
int tb_set_vecnorm(tb_ctx *ctx, const tb_vecnorm *cfg, const double *d_stats, void *stream);
/* One record per agent: `agents` records of one configuration cfg.  d_stats double [agents, TB_VECNORM_WORDS(obs_dim)]: the
 * records to start from (NULL: all fresh); each row is checked as tb_set_vecnorm checks its record, and a failure names the
 * row; with d_stats the call synchronises `stream`.  agents >= 1 must divide N; agents = 1 is tb_set_vecnorm, with its kernels
 * and launches, and cfg NULL detaches.  Zeroes the returns of all N envs and arms the reset fold (one launch).  A call that
 * needs more records or partials than the buffers hold allocates larger ones (cudaMalloc, and cudaFree of the old ones, which
 * waits for the device): as with tb_set_policies, make the largest call before capturing, and capture again after a call that
 * grew them.  A rejected call leaves the context as it was. */
int tb_set_vecnorms(tb_ctx *ctx, const tb_vecnorm *cfg, int64_t agents, const double *d_stats, void *stream);
/* d_stats double [TB_VECNORM_WORDS(obs_dim)] = the current record (stream-ordered copy, never synchronises).  Fails when no
 * normaliser is attached, and when more than one record is (tb_get_vecnorms reads them). */
int tb_get_vecnorm(tb_ctx *ctx, double *d_stats, void *stream);
/* d_stats double [agents, TB_VECNORM_WORDS(obs_dim)] = every record (stream-ordered copy, never synchronises).  Fails when no
 * normaliser is attached or agents is not the number of records attached. */
int tb_get_vecnorms(tb_ctx *ctx, double *d_stats, int64_t agents, void *stream);
/* The library's record buffer, double [*agents, TB_VECNORM_WORDS(obs_dim)], and the number of records attached.  The kernels
 * read a record when they run, so a stream-ordered write into a row (a PBT copy of one agent's record over another's) is seen
 * by the next kernel that reads it, a replayed graph included; unlike tb_set_vecnorms it zeroes no return and arms no fold.
 * The pointer stays valid until a tb_set_vecnorms call grows the buffer or the context is destroyed.  Fails when no normaliser
 * is attached. */
int tb_vecnorm_device_ptr(tb_ctx *ctx, double **d_records, int64_t *agents);
/* d_out = rule 4's o^ of d_in float32 [rows, obs_dim] (what = TB_VECNORM_OBS), or rule 3's r^ of d_in float32 [rows]
 * (TB_VECNORM_REWARD), with the record as it stands when the kernel runs (a replayed graph sees the current statistics);
 * norm_obs = 0 (norm_reward = 0) copies.  What SB3's ReplayBuffer.sample(env=vec_normalize_env) does to a raw batch.  d_out
 * may be d_in.  One kernel launch (rows = 0 included, which reads nothing), never synchronises.  Fails when no normaliser is
 * attached, what is unknown, rows < 0 (or the grid would exceed 2^31 - 1 CTAs of 128 floats), d_in or d_out is NULL while
 * rows > 0, or the context is faulted, or more than one record is attached (tb_set_vecnorms). */
#define TB_VECNORM_OBS 0
#define TB_VECNORM_REWARD 1
int tb_vecnorm_apply(tb_ctx *ctx, const float *d_in, int64_t rows, int what, float *d_out, void *stream);

/* ---- ES fitness rollout (SURVEY 8(f)-2): fitness_static (fitness_functions.py:18-158) for a whole population in one context.
 * Env i evaluates individual i / (N / individuals) with the reference's GatedCNN (policies.py:59-128) on an 8-step history of
 * observations, each normalised by the env's own float64 running normaliser (evolution_strategy_static.py:25-44); the
 * action is clipped to [-1, 1].  Parameters per individual, float32, in parameters_to_vector order (each conv weight
 * [out][in][2]):
 *   conv_0 W[8 x C x 2] b[8], conv_gate_0 W[8 x C x 2] b[8]          (dilation 1)
 *   conv_1 W[12 x 8 x 2] b[12], conv_gate_1 W[12 x 8 x 2] b[12]      (dilation 2)
 *   conv_2 W[A x 12 x 2] b[A]                                       (dilation 4)
 * with C = obs_dim, A = act_dim: 766 floats for SwingRacket-v0, 858 for Tennisbot-v0. */
#define TB_ES_FLOATS 766
#define TB_ES_FLOATS_HIT 858
#define TB_ES_HISTORY 8
int tb_es_floats(int env_kind); /* TB_ES_FLOATS / TB_ES_FLOATS_HIT (-1: unknown kind); callable without a GPU */
/* Start a generation: d_weights float32 [individuals, floats] (floats = tb_es_floats(env_kind), individuals must divide N; the
 * library keeps its own copy, so the buffer may be reused once the stream has passed this call); d_normalizer double
 * [3, obs_dim] = the master normaliser's (n, mean, mean_diff), NULL = zeros.  Resets every env from the RNG (a context's first
 * generation places as tb_reset does on a fresh context; later generations continue the episode counters), observes the reset
 * observation, fills the history with its normalised value, zeroes the returns and marks every env alive.  Needs
 * TB_CONTROL_FORCE.  Stream-ordered, never synchronises. */
int tb_es_begin(tb_ctx *ctx, const float *d_weights, int64_t individuals, int64_t floats, const double *d_normalizer,
                void *stream);
/* k_steps >= 1 env steps of the generation: per step one es_kernel launch (fold the previous step's reward, done and observation
 * into return, alive, normaliser and history; GatedCNN forward) and tb_step's launches, then one fold-only es_kernel launch.
 * return += reward while alive, then alive &= !done; after an env's first done it acts 0 and its normaliser and history stop.
 * d_return double [N], d_alive uint8 [N] (required): the state after the last step.  Optional traces (NULL = none):
 * d_obs float32 [K + 1, N, obs_dim], the raw observation the normaliser consumed before each action (the terminal one when the
 * step ended an episode; [0] is the one consumed before this call, [K] the last step's); d_actions float32 [K, N, act_dim], the
 * clipped actions; d_reward float32 [K, N]; d_done uint8 [K, N].  The envs must not be stepped by other calls between
 * tb_es_begin and the last tb_es_rollout of a generation.  Never synchronises: capturable in a CUDA graph. */
int tb_es_rollout(tb_ctx *ctx, int k_steps, double *d_return, uint8_t *d_alive, float *d_obs, float *d_actions,
                  float *d_reward, uint8_t *d_done, void *stream);

/* ---- ES population and update (ARS V2-t with seeded perturbations).  Direction j's noise in generation g is a float32 vector
 * eps_j drawn from Philox, so any shard can regenerate it:
 *   r = Philox4x32-10(key = noise_seed, counter = (j lo, j hi, g, (3 << 28) | ((f / 4) << 4))),  q = f / 4, k = 0, 1:
 *   u1 = (r[2k] + 0.5) / 2^32, u2 = r[2k + 1] / 2^32, rho = sqrt(-2 ln u1) (float64),
 *   eps_j[4q + 2k] = float32(rho cos(2 pi u2)), eps_j[4q + 2k + 1] = float32(rho sin(2 pi u2)).
 * Global individual g = env_id_offset / repeats + p (p local) belongs to direction j = g / 2 and is theta + d for even g,
 * theta - d for odd g, with d = float32(sigma * eps_j) and one float32 rounding per add (no fused multiply-add).
 * tb_es_begin_noise is tb_es_begin with that population drawn in the library from d_theta float32 [floats]; it also fails when
 * individuals is odd, env_id_offset is not a multiple of 2 x repeats (a shard holds whole pairs), sigma is not a finite number
 * above 0 or d_theta is NULL.  Stream-ordered, never synchronises. */
int tb_es_begin_noise(tb_ctx *ctx, const float *d_theta, int64_t individuals, int64_t floats, float sigma, uint64_t noise_seed,
                      uint32_t generation, const double *d_normalizer, void *stream);
/* d_out float32 [tb_es_floats(env_kind)] = sum_k d_coef[k] * eps_{d_dirs[k]} of generation `generation`, accumulated in float64 in
 * the order k = 0 .. count - 1 and rounded once.  d_dirs int64 [count] are global direction indices, d_coef float32 [count];
 * count may be 0 (d_out = 0).  Stream-ordered, never synchronises. */
int tb_es_noise_combine(tb_ctx *ctx, const int64_t *d_dirs, const float *d_coef, int64_t count, uint64_t noise_seed,
                        uint32_t generation, float *d_out, void *stream);
/* d_out double [3, obs_dim] = (count, mean, M2) of the observations this context's normalisers took since the last
 * tb_es_begin* (the master's share excluded): each env's reset observation and one per step until its first done (the
 * terminal observation is not taken).  Combine shards and the master with Chan's formula.  A deterministic two-pass
 * reduction, no atomics.  Fails before the first tb_es_begin*.  Stream-ordered, never synchronises. */
int tb_es_normalizer_stats(tb_ctx *ctx, double *d_out, void *stream);

/* ---- SAC actor and replay ring (SURVEY 8(f)-5): what SB3 SAC's collect_rollouts does around env.step (train_swing.py's and
 * train.py's SAC option), kept on the device.  The actor is SB3 1.8 SAC MlpPolicy's: latent_pi = Linear(obs, 256), ReLU,
 * Linear(256, 256), ReLU; heads mu and log_std = Linear(256, act); log_std clamped to [-20, 2]; action = tanh(mu + exp(log_std)
 * eps) (TB_SAC_SAMPLE) or tanh(mu) (TB_SAC_MEAN).  Both action spaces are Box(-1, 1), so SB3's unscaling is the identity.
 * Parameters, float32, in SB3 state-dict order, each tensor row-major [out][in] and padded to a multiple of 4 floats:
 *   actor.latent_pi.0 W[256 x obs] b[256], actor.latent_pi.2 W[256 x 256] b[256], actor.mu W[act x 256] b[act],
 *   actor.log_std W[act x 256] b[act]:  70672 floats for SwingRacket-v0 (obs 6, act 6), 70152 for Tennisbot-v0 (obs 12, act 2).
 * Numerics: layer 1 in float32 (each product and sum rounded, in input order, starting from the bias), ReLU, rounded to BF16;
 * layer 2 on the tensor cores with W2 rounded to BF16 and FP32 accumulation; b2, ReLU, the heads, exp and tanh in float32.
 * Noise: r = Philox4x32-10(key = noise_seed, counter = (global env id lo, hi, tick, (4 << 28) | q)), q = o / 4, where tick is
 * the context's env-step counter when the action is taken (so every replay of a captured graph draws fresh noise, and
 * shards reproduce the full batch).  With v(x) = (x >> 8) / 2^24:
 *   TB_SAC_UNIFORM: action[o] = 2 v(r[o mod 4]) - 1 (SB3's learning_starts warm-up; the network is not evaluated);
 *   TB_SAC_SAMPLE: pair p = o / 2 of words w = r[(2p) mod 4], r[(2p + 1) mod 4]: u1 = v(w0) + 2^-25, u2 = v(w1),
 *     eps[o] = sqrtf(-2 logf(u1)) * (o even ? cospif(2 u2) : sinpif(2 u2)), all float32. */
#define TB_SAC_FLOATS 70672
#define TB_SAC_FLOATS_HIT 70152
#define TB_SAC_HIDDEN 256
#define TB_SAC_SAMPLE 0
#define TB_SAC_MEAN 1
#define TB_SAC_UNIFORM 2
int tb_sac_floats(int env_kind); /* TB_SAC_FLOATS / TB_SAC_FLOATS_HIT (-1: unknown kind); callable without a GPU */
/* Converts d_params (count = tb_sac_floats(env_kind)) on the device into the library's own image of the actor (W2 as BF16 in
 * the tensor cores' shared-memory layout): one kernel on `stream`, so it is capturable and a replayed graph sees the weights the
 * buffer holds at replay time.  Returns the context to one actor after tb_set_sac_actors. */
int tb_set_sac_actor(tb_ctx *ctx, const float *d_params, int64_t count, void *stream);
/* A population of SAC actors for one context: d_params float32 [agents, tb_sac_floats(env_kind)], rows in tb_set_sac_actor's
 * layout; env i acts with actor i / (N / agents).  One kernel launch converts every row into the library's image, stream-ordered
 * like tb_set_sac_actor: capturable, and a replayed graph converts the weights d_params holds at replay time.  A call with more
 * agents than the image buffer holds allocates a larger one (cudaMalloc, and cudaFree of the old one, which waits for the
 * device): make the largest call before capturing, and capture again after a call that grew the buffer, since graphs captured
 * earlier refer to the old one.  Fails on a NULL d_params, agents < 1, agents not dividing N, count != agents x
 * tb_sac_floats(env_kind), a faulted context, and, for agents > 1, N / agents not a multiple of 128 (a 128-env tile of
 * sac_kernel multiplies against one W2 image in shared memory, and two 128 KB images do not fit beside its A tile).  A
 * rejected call leaves the actors as they were.  agents = 1 is tb_set_sac_actor (the same image and launch). */
int tb_set_sac_actors(tb_ctx *ctx, const float *d_params, int64_t agents, int64_t count, void *stream);
/* Replay ring, caller-owned device arrays: obs, next_obs float32 [slots, N, obs_dim]; act float32 [slots, N, act_dim]; reward
 * float32 [slots, N]; done uint8 [slots, N]. */
typedef struct tb_sac_ring {
  uint32_t struct_size; /* sizeof(tb_sac_ring) */
  int32_t reserved;
  int64_t slots;
  float *obs, *act, *reward, *next_obs;
  uint8_t *done;
} tb_sac_ring;
/* Needs TB_CONTROL_FORCE and auto_reset = 1.  Resets every env from the RNG, keeps the reset observation in the context and
 * records the env-step counter as the ring's base.  One kernel launch. */
int tb_sac_begin(tb_ctx *ctx, void *stream);
/* k_steps >= 1 env steps: per step one sac_kernel launch (fold the previous step into the ring, then act) and tb_step's
 * launches, then one fold-only sac_kernel launch: (K + 1) + K s launches, s = 2 for SwingRacket-v0 and 1 for Tennisbot-v0.
 * The j-th env step since tb_sac_begin writes ring slot j mod slots (j is read on the device, so a captured graph appends at
 * new slots on every replay): obs = the observation the action was computed from, act = the squashed action step_kernel
 * received, reward, done (a time-out is a done like any other: the reference returns {} and SB3 does not bootstrap), next_obs
 * = the terminal observation when done, else the step's observation.  ring = NULL stores nothing (evaluation).  d_last_obs
 * float32 [N, obs_dim] (may be NULL) receives the observation after the last step.  mode TB_SAC_SAMPLE and TB_SAC_MEAN need
 * tb_set_sac_actor.  Never synchronises: capturable in a CUDA graph.
 * After tb_set_sac_actors with agents P > 1, env i acts with actor i / n, n = N / P; the ring's layout, the noise keys,
 * d_last_obs and the launch count stay as they are (TB_SAC_UNIFORM ignores the actors).  Agent p's transitions are columns
 * [p n, (p + 1) n) of every ring slot, and agent p's envs give, bit for bit, what a context of n envs with env_id_offset = p n
 * and the same seed gives with tb_set_sac_actor(row p): actions, ring columns and d_last_obs.
 * mode | TB_SAC_VECNORM (fails when no normaliser is attached, when more than one record is, and when more than one actor is set,
 * naming the counts): SB3 SAC under VecNormalize, with the normaliser of tb_set_vecnorm.
 * After every env step (TB_SAC_UNIFORM included) a training normaliser folds the step's observation of all N envs (rule 1),
 * the return (rule 2) and zeroes the returns of done envs (rule 3); the actor acts on o^ (rule 4) with the statistics after
 * that fold.  The ring, d_last_obs and tb_read_stats stay RAW (SB3's get_original_obs / get_original_reward; a terminal
 * next_obs is the exact raw value, where SB3 stores unnormalize(normalize(.)), which differs where clip_obs bites).  The first
 * such rollout with a training normaliser after tb_sac_begin zeroes the returns and folds the reset observation of all envs
 * (a flag of tb_sac_begin, kept on the device); training = 0: statistics and returns never change.  Launches: (K + 1) + K s
 * frozen; training adds 2 K (the statistics pass after each step) + 3 (the entry pass, which folds only while the reset is
 * pending). */
#define TB_SAC_VECNORM 0x100
int tb_sac_rollout(tb_ctx *ctx, int k_steps, int mode, uint64_t noise_seed, const tb_sac_ring *ring, float *d_last_obs,
                   void *stream);

/* ---- frames rendered on the device: one ray per pixel against the scene's collision shapes.  No GUI; the reference's
 * PyBullet camera (tennisbot_env.py:269-279) is not recorded, so cameras are the caller's.
 *
 * Geometry: the collision shapes as the physics sees them, without the collision margins (hull_margin, box_margin), all in
 * the world frame (metres):
 *   TB_BODY_COURT   the floor box |x| <= floor_hx, |y| <= floor_hy, |z| <= floor_hz (centred on the origin, as physics_step has it);
 *   TB_BODY_NET     the net box   |x| <= net_hx,   |y| <= net_hy,   |z| <= net_hz;
 *   TB_BODY_GOAL    SwingRacket-v0 contexts only (the hit env has no goal): the goal prism, the 32-gon of goal_vertex_x/y
 *                   (tb_scene_constant) about the record's goal x, y (TB_S_GOAL), |z| <= goal_half_z;
 *   TB_BODY_RACKET  the racket's outline prism in its COM frame: |x| <= racket_scale * racket_half_x, polygon (y, z) =
 *                   racket_scale * (racket_outline_y, racket_outline_z - racket_com_z); placed at the record's COM position
 *                   (TB_S_RACKET_POS) and quaternion (TB_S_RACKET_QUAT, x,y,z,w, used as the physics uses it: unnormalised);
 *                   the convex hull the physics uses, not the STL mesh;
 *   TB_BODY_BALL    the sphere of radius ball_radius at TB_S_BALL_POS.
 * The context's current scene is used, so racket_scale applies.  There are no court lines (the court texture is not part of
 * this repository).  A shape is seen where the ray enters it at a positive distance (an eye inside a shape does not see it);
 * the nearest entry wins, equal distances go to the lower TB_BODY_* value.
 * Camera: f = normalize(target - eye), r = normalize(f x up), u = r x f, t = tan(fov_y / 2).  Pixel (x, y), x = column,
 * y = row with row 0 at the top (gym's rgb_array layout), casts the ray direction
 *   d = normalize(f + ((2 (x + 0.5) / W - 1) t W / H) r + ((1 - 2 (y + 0.5) / H) t) u).
 * Shading: n = the unit outward normal of the surface the ray enters (for a box or a prism: the entry plane's), flipped to
 * face the eye (n.d <= 0); channel k = floor(c_body[k] (0.35 + 0.65 max(0, n.L)) + 0.5) with L = TB_RENDER_LIGHT
 * normalised; a ray that meets nothing gets TB_RENDER_SKY.  No shadows, no anti-aliasing.  The kernel computes in float32
 * with coordinates relative to the eye (the per-frame plane offsets in float64, rounded once). */
#define TB_BODY_NONE 0
#define TB_BODY_COURT 1 /* the floor box */
#define TB_BODY_NET 2
#define TB_BODY_GOAL 3  /* SwingRacket-v0 only */
#define TB_BODY_RACKET 4
#define TB_BODY_BALL 5
#define TB_RENDER_SKY {170, 200, 235}
#define TB_RENDER_COLORS {{0, 0, 0}, {70, 140, 95}, {235, 235, 235}, {215, 60, 50}, {40, 80, 200}, {225, 240, 60}} /* by TB_BODY_* */
#define TB_RENDER_LIGHT {-0.3, 0.4, 1.0} /* towards the light, before normalisation */
#define TB_RENDER_MAX_SIZE 4096
typedef struct tb_camera {
  uint32_t struct_size;            /* sizeof(tb_camera) */
  int32_t width, height;           /* pixels, 1 .. TB_RENDER_MAX_SIZE each */
  int32_t reserved;
  double eye[3], target[3], up[3]; /* world frame, metres */
  double fov_y_deg;                /* vertical field of view, (0, 180) */
} tb_camera;
/* d_states double [count, TB_STATE_WORDS]: canonical records (tb_get_state rows, a trajectory file, or the caller's).
 * d_rgb uint8 [count, H, W, 3]; d_depth float32 [count, H, W], the distance from the eye along the ray, +inf where the ray
 * meets nothing (may be NULL); d_body uint8 [count, H, W], TB_BODY_* (may be NULL).  One kernel launch on `stream`, never
 * synchronises (capturable in a CUDA graph).  Reads only the context's scene parameters and writes nothing of the context
 * (env state, RNG counters, statistics and fast-forward queues are untouched; tb_launch_count rises by 1).  Fails when cam,
 * d_states or d_rgb is NULL, count < 1, struct_size is wrong, width or height is outside 1 .. 4096, fov_y_deg is not finite
 * or outside (0, 180), eye == target, up is parallel to the view direction (|f x up| <= 1e-9 |up|, a zero up included), an
 * output's size in bytes overflows int64, or the context is faulted. */
int tb_render(tb_ctx *ctx, const tb_camera *cam, const double *d_states, int64_t count, uint8_t *d_rgb, float *d_depth,
              uint8_t *d_body, void *stream);

/* ---- one env step traced substep by substep: what tb_step does to a record, with the record kept after every physics
 * substep.  SwingRacket-v0's 26th step fast-forwards the ball's whole flight inside one env step; the trace shows it (pass
 * trace rows to tb_render for frames of the flight).
 * Bound: a step stops after its first substep when that substep's step counter k (the counter after it) is <= 25 or the env
 * is done (phase 0); otherwise it runs until a landing or the time-out k > 800, which ends it at k = 801 at the latest.  So a
 * step that starts from a step counter s0 >= 25 takes at most max(801 - s0, 2) <= 801 - 25 = 776 substeps, and any smaller s0
 * takes 1.  Tennisbot-v0's step is always one substep. */
#define TB_TRACE_MAX_SUBSTEPS 776
int tb_trace_max_substeps(int env_kind); /* TB_TRACE_MAX_SUBSTEPS for SwingRacket-v0, 1 for Tennisbot-v0, -1 unknown; no GPU needed */
/* d_states double [count, TB_STATE_WORDS]: canonical records from any source (copies: the context's envs are not involved);
 * d_actions float32 [count, act_dim], the actions as tb_step receives them (clipping to the Box is the caller's job).
 * d_trace double [max_substeps, count, TB_STATE_WORDS]: [k, i] is record i after substep k + 1.  The step counter advances every
 * substep; the return and the done bit change at the final substep only, as tb_step leaves them.  Records from substeps up to
 * max_substeps - 1 repeat the final record, which is the terminal state (no auto-reset: what tb_get_state shows after tb_step
 * with auto_reset = 0).  A step longer than max_substeps stores its first max_substeps records and still runs to its end.
 * d_bits uint8 [max_substeps, count] (may be NULL): the contact bits of that substep alone, TB_EV_RACKET_BALL | COURT_BALL |
 * GOAL_BALL | NET_BALL | RACKET_LOW; 0 in the repeated records.  d_substeps int32 [count]: substeps the step took.
 * d_reward float32, d_done uint8, d_events uint8, each [count] (may be NULL): what tb_step returns for that record and action
 * (events: the OR of the substep bits, plus TB_EV_TIMEOUT / TB_EV_BALL_PASSED).  The kernel computes in the context's
 * precision, reads only its scene parameters and writes nothing of the context.  One kernel launch on `stream`, never
 * synchronises (capturable in a CUDA graph).  Fails when d_states, d_actions, d_trace or d_substeps is NULL, count < 1,
 * max_substeps is outside 1 .. tb_trace_max_substeps(env_kind), the context is in TB_CONTROL_PID (its controller memory is
 * not part of the record), count x max_substeps x 256 bytes overflows int64, or the context is faulted. */
int tb_trace_step(tb_ctx *ctx, const double *d_states, const float *d_actions, int64_t count, int32_t max_substeps,
                  double *d_trace, uint8_t *d_bits, int32_t *d_substeps, float *d_reward, uint8_t *d_done,
                  uint8_t *d_events, void *stream);

/* ---- state dump / injection for the parity harness: double [N, TB_STATE_WORDS] */
int tb_get_state(tb_ctx *ctx, double *d_state, void *stream);
int tb_set_state(tb_ctx *ctx, const double *d_state, void *stream);

/* ---- episode statistics, accumulated in-kernel (warp reductions + one atomic per warp) */
int tb_stats_device_ptr(tb_ctx *ctx, int64_t **d_stats); /* int64 [TB_NUM_STATS] in HBM: all-reduce this over NCCL */
int tb_read_stats(tb_ctx *ctx, int64_t *h_stats, int clear, void *stream); /* synchronises `stream` */

/* ---- host-buffer convenience (what a numpy VecEnv calls): one env step with the actions taken from and the results left in
 * HOST arrays, on the context's own stream, synchronised before returning.  Transport, by default: when every buffer is
 * pinned (cudaHostAlloc / torch pin_memory) the kernels address the host buffers themselves - actions are read and results
 * written over PCIe while the step computes, both directions at once (zero copy); pageable buffers are staged (H2D copy,
 * kernels, D2H copies).  TB_HOST_MODE=staging stages pinned buffers too (eight GPUs stepping at once were faster staged,
 * DESIGN.md section 4); TB_HOST_MODE=zero_copy or unset is the default above, and any other value makes the call fail.
 * A call also fails if a fast-forward launch of the context has timed out (see tb_ff_diagnostics). */
int tb_reset_host(tb_ctx *ctx, const uint8_t *h_mask, float *h_obs);
int tb_step_host(tb_ctx *ctx, const float *h_actions, float *h_obs, float *h_reward, uint8_t *h_done,
                 float *h_terminal_obs, uint8_t *h_events);

/* number of kernels this context has launched, tb_create's and tb_set_param's included (bench.py's gpu_launches) */
int tb_launch_count(tb_ctx *ctx, int64_t *launches);

/* Diagnostics of the most recent SwingRacket fast-forward (the launch of tb_step's second kernel on an env's 26th
 * step; read it before the next step): out[0] = 1 if one ran, out[1] = visits of envs to the generic full-substep path
 * (server warps), out[2] = nanoseconds until every flight had landed, out[3..14] = 0 (reserved; the finishing pass
 * overlaps the flights, so it has no time of its own), out[15] = non-zero if a wait inside a fast-forward
 * launch of this context has ever timed out (sticky; that launch left envs unfinished instead of hanging the device, and
 * EVERY later call on the context - tb_step, tb_step_host, tb_reset, tb_rollout, tb_read_stats - fails from then on: the
 * fault word is mirrored in mapped host memory and checked on entry without synchronising).  A wait gives up after
 * TB_FF_SPIN_LIMIT_MS (default 4000 ms).  ff_kernel has no grid barrier and claims all of its work from counters and queues,
 * so it completes whatever else occupies SMs while it runs; the time-out is the backstop.  Synchronises the device.
 * h_out: 16 x int64. */
int tb_ff_diagnostics(tb_ctx *ctx, int64_t *h_out);

/* Per-kernel device timing for roofline reports.  While enabled, every tb_step brackets its two kernels with CUDA
 * events on the launch stream and synchronises the stream to accumulate their durations (so do not enable it
 * inside a throughput measurement).  tb_get_kernel_timing returns the accumulated milliseconds of step_kernel and
 * ff_kernel and the number of steps they cover, and clears the accumulators. */
int tb_set_kernel_timing(tb_ctx *ctx, int enabled);
int tb_get_kernel_timing(tb_ctx *ctx, double *ms_step_kernel, double *ms_ff_kernel, int64_t *steps);

#ifdef __cplusplus
}
#endif
#endif

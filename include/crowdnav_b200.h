/*
 * crowdnav_b200.h -- C ABI of libcrowdnav_b200.so (sm_100a).
 *
 * Drop-in boundary for the data-parallel hot path of minh86/ModelCrowdNav: the CrowdSim
 * environment step (ORCA humans, kinematics, collision/discomfort, reward/done) and the
 * SARL / MultiHumanRL one-step lookahead, batched over E independent environments that live
 * in HBM as a struct-of-arrays.  Plain pointers and sizes only; no torch types.
 *
 * Every entry point names the reference interface it replaces (file:line relative to the
 * reference repository root).  All functions return 0 (CN_OK) or a negative CN_E* code;
 * cn_last_error() gives the thread-local message.  One handle per GPU per process, not
 * thread-safe.  `stream` arguments are cudaStream_t passed as void* (0 = default stream; pass
 * torch.cuda.current_stream().cuda_stream); nothing synchronises except the functions
 * documented as blocking (host getters).  There is NO CPU fallback: every compute entry point
 * fails with CN_ECUDA when no sm_100 device is usable.
 */
#ifndef CROWDNAV_B200_H
#define CROWDNAV_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CN_OK 0
#define CN_EINVAL (-1)
#define CN_ECUDA (-2)
#define CN_ENOMEM (-3)
#define CN_EUNSUPPORTED (-4)
#define CN_EVALUE (-5) /* "Value network is not well trained." (multi_human_rl.py:57-58) */

#define CN_AGENT_STRIDE 8     /* px py vx vy gx gy radius v_pref */
#define CN_MAX_NEIGHBORS 16   /* ORCA max_neighbors supported by the kernel (reference: 10) */
#define CN_MAX_HUMANS 64
/* Robot kinematics.  HOLONOMIC: ActionXY (vx, vy) -- [action_space] kinematics = holonomic.  UNICYCLE: ActionRot (v, r),
 * r in [-pi/4, pi/4], robot heading theta in the state and in rotate().  NONE: the fork exactly as shipped -- cadrl.py:66
 * comments the config read out, so policy.kinematics stays None: ActionRot dynamics (every `== 'holonomic'` test fails)
 * while rotate() leaves the heading feature at zero (its test is `== 'unicycle'`). */
#define CN_KIN_HOLONOMIC 0
#define CN_KIN_UNICYCLE 1
#define CN_KIN_NONE 2
#define CN_MAX_ACTIONS 128

/* info codes = crowd_sim/envs/utils/info.py:1-38 */
enum { CN_NOTHING = 0, CN_DANGER = 1, CN_REACHGOAL = 2, CN_COLLISION = 3, CN_TIMEOUT = 4 };
/* scene rules = crowd_sim.py:105-112 */
enum { CN_CIRCLE_CROSSING = 0, CN_SQUARE_CROSSING = 1 };
/* value-network arithmetic */
enum { CN_PREC_F32 = 0 /* FP32 CUDA cores */, CN_PREC_F16_TC = 1 /* fp16 operands, fp32 accumulate, tcgen05 */ };
enum { CN_NET_SARL = 0, CN_NET_CADRL = 1, CN_NET_LSTM_RL = 2 };   /* value network behind the lookahead */
enum { CN_WORLD_ATTENTION = 0, CN_WORLD_MLP = 1 };                /* learned human-motion model (world_model.py) */

typedef struct cn_env cn_env;
typedef struct cn_policy cn_policy;

/* CrowdSim.configure (crowd_sim.py:58-89) + ORCA.__init__ (orca.py:55-67) + agent attributes
 * (agent.py:16-18), flattened.  Use cn_env_cfg_default() then override. */
typedef struct {
    int32_t num_envs;            /* E: environments resident on this GPU */
    int32_t human_num;           /* H ([sim] human_num) */
    double time_limit;           /* [env] time_limit = 25 */
    double time_step;            /* [env] time_step = 0.25 */
    double success_reward;       /* [reward] */
    double collision_penalty;
    double discomfort_dist;
    double discomfort_penalty_factor;
    double neighbor_dist;        /* orca.py:61 */
    int32_t max_neighbors;       /* orca.py:62 */
    double time_horizon;         /* orca.py:63 */
    double human_safety_space;   /* orca.py:60 */
    int32_t robot_visible;       /* [robot] visible */
    /* device-side reset (throughput runs; parity runs upload host scenes with cn_env_set_state) */
    int32_t sim_rule;            /* CN_CIRCLE_CROSSING / CN_SQUARE_CROSSING */
    double circle_radius;        /* [sim] circle_radius = 4 */
    double square_width;         /* [sim] square_width = 10 */
    double human_radius, human_v_pref, robot_radius, robot_v_pref;
    uint64_t seed;               /* Philox key */
    int64_t env_id_offset;       /* global id of env 0 (rank * E): results do not depend on the GPU count */
    int32_t auto_reset;          /* 1: an env that finished an episode is re-generated at the end of the step */
    double gamma;                /* [rl] gamma, for the per-episode discounted return (explorer.py:124-125) */
    int32_t randomize_attributes; /* [env] randomize_attributes: device resets draw v_pref ~ U(0.5,1.5) and radius ~
                                   * U(0.3,0.5) per human before placing it (crowd_sim.py:167-168, agent.py:39-45) */
    int32_t robot_kinematics;    /* CN_KIN_*: how CrowdSim.step reads the robot action (crowd_sim.py:350-354, agent.py:110-135) */
} cn_env_cfg;

/* SARL.configure (sarl.py:73-86) + CADRL.set_common_parameters (cadrl.py:64-73) */
typedef struct {
    int32_t input_dim;           /* 13 (cadrl.py:53-55) */
    int32_t self_state_dim;      /* 6 */
    int32_t mlp1_dims[2];        /* 150,100 */
    int32_t mlp2_dims[2];        /* 100,50 */
    int32_t attn_dims[3];        /* 100,100,1 */
    int32_t mlp3_dims[4];        /* 150,100,100,1 */
    int32_t speed_samples;       /* 5 */
    int32_t rotation_samples;    /* 16 */
    double gamma;                /* 0.9 */
    double v_pref;               /* robot v_pref used to build the action table (cadrl.py:147) */
    int32_t precision;           /* CN_PREC_* */
    int32_t kinematics;          /* CN_KIN_*: action space of CADRL.build_action_space (cadrl.py:82-102) and the theta
                                  * feature of rotate() (cadrl.py:236-240); must equal the env's robot_kinematics */
    /* Which value network sits behind the lookahead (policy_factory: sarl, cadrl, lstm_rl).  CN_NET_CADRL
     * (cadrl.py:22-30,131-178): mlp3_dims = [cadrl] mlp_dims applied to every (robot, human) row, value = reward +
     * gamma_bar * MIN over humans.  CN_NET_LSTM_RL (lstm_rl.py:9-105): humans sorted by decreasing distance (query_env =
     * false only, see multi_human_rl.py:37-42), nn.LSTM(13 or lstm_mlp1_dims[3] -> lstm_hidden) over the rows, mlp3_dims =
     * [lstm_rl] mlp2_dims on cat(self_state, h_n); lstm_mlp1_dims[0] > 0 selects ValueNetwork2 (with_interaction_module).
     * Both run on either precision: CN_PREC_F16_TC takes the reference's default shapes (CADRL mlp_dims 150,100,100,1; LSTM-RL
     * without interaction module / occupancy maps, lstm_hidden 50, mlp2_dims 150,100,100,1), CN_PREC_F32 any shape. */
    int32_t network;             /* CN_NET_* */
    int32_t lstm_hidden;         /* [lstm_rl] global_state_dim = 50 */
    int32_t lstm_mlp1_dims[4];   /* [lstm_rl] mlp1_dims = 150,100,100,50; {0} = ValueNetwork1 */
    /* Occupancy maps ([sarl] / [lstm_rl] with_om = true, multi_human_rl.py:43-50,98-163): every rotated row is followed by
     * the cell_num x cell_num x om_channel_size map of the OTHER humans around that human, built once per lookahead from
     * the next human states; input_dim must be 13 + cell_num^2 * om_channel_size.  SARL: both precisions (on the tensor-core
     * path the map, which does not depend on the action, enters mlp1.0 as one fp32 row bias per human); LSTM-RL: FP32. */
    int32_t with_om;
    int32_t cell_num;            /* [om] cell_num = 4 (<= 8) */
    double cell_size;            /* [om] cell_size = 1 */
    int32_t om_channel_size;     /* [om] om_channel_size = 3 (1, 2 or 3) */
    /* [sarl] with_global_state = false: attention.0 reads mlp1_out only (sarl.py:40-47), so its weight is
     * [attn_dims[0]][mlp1_dims[1]] instead of [attn_dims[0]][2 * mlp1_dims[1]]; 0 = the reference default.  SARL only (with or
     * without occupancy maps, both precisions); CN_EINVAL for CADRL and LSTM-RL. */
    int32_t without_global_state;
} cn_sarl_cfg;

/* Episode statistics accumulated on the device by cn_env_step(update=1); the counters
 * Explorer.run_k_episodes keeps (explorer.py:41-51,92-108,124-141). */
typedef struct {
    int64_t episodes, success, collision, timeout;
    int64_t steps;               /* env steps taken (update=1) */
    int64_t too_close;           /* Danger steps */
    double sum_min_dist;         /* sum of Danger.min_dist */
    double sum_success_time, sum_collision_time, sum_timeout_time;
    double sum_return;           /* sum over finished episodes of sum_t gamma^(t*dt*v_pref) r_t */
} cn_stats;

const char *cn_last_error(void);
int cn_version(void);
int cn_device_count(void);

void cn_env_cfg_default(cn_env_cfg *cfg);   /* values of crowd_nav/configs/env.config */
void cn_sarl_cfg_default(cn_sarl_cfg *cfg); /* values of crowd_nav/configs/policy.config */

/* ---- environment: replaces gym.make('CrowdSim-v0') + configure (crowd_sim.py:19-89) ---- */
int cn_env_create(const cn_env_cfg *cfg, int device, cn_env **out);
int cn_env_destroy(cn_env *env);

/* CrowdSim.reset with host-generated scenes (crowd_sim.py:261-323).  agents: E x (H+1) x 8 doubles
 * (agent 0 = robot), times: E doubles or NULL (= 0).  Clears per-episode accumulators. */
int cn_env_set_state(cn_env *env, const double *agents_host, const double *times_host, void *stream);
/* Blocking read-back in the same layout. */
int cn_env_get_state(cn_env *env, double *agents_host, double *times_host, void *stream);
/* Robot heading (FullState.theta), E doubles.  Resets and cn_env_set_state put it at pi/2 (crowd_sim.py:284); the
 * non-holonomic step wraps it to [0, 2 pi) (agent.py:131).  Only read when robot_kinematics != CN_KIN_HOLONOMIC. */
int cn_env_set_theta(cn_env *env, const double *theta_host, void *stream);
int cn_env_get_theta(cn_env *env, double *theta_host, void *stream);
/* CrowdSim.reset on the device (crowd_sim.py:165-217 distributions and rejection rule, Philox stream
 * keyed by (seed, global env id, episode counter)) for every env of the handle. */
int cn_env_reset(cn_env *env, void *stream);

/* Human ORCA actions for the current state: replaces the rvo2.PyRVOSimulator traffic of
 * ORCA.predict (orca.py:82-132) for every human of every env (crowd_sim.py:337-342).  The result is
 * cached on the device and reused by cn_env_step and cn_policy_lookahead (query_env). */
int cn_env_orca(cn_env *env, void *stream);
/* Robot action from an ORCA policy (imitation learning, train.py:157-166): writes the env's
 * pending action. */
int cn_env_robot_orca(cn_env *env, double safety_space, void *stream);

/* CrowdSim.step(action, update) / onestep_lookahead (crowd_sim.py:325-434).  action_xy_dev: device
 * pointer E x 2 doubles, or NULL to use the pending action chosen by cn_policy_lookahead /
 * cn_env_robot_orca.  Requires cn_env_orca for the current state. update=0 leaves the state untouched
 * and fills next_obs. */
int cn_env_step(cn_env *env, const double *action_xy_dev, int update, void *stream);

/* Device views of the last step's outputs (valid until the next call that writes them). */
typedef struct {
    const double *reward;      /* E */
    const uint8_t *done;       /* E */
    const uint8_t *info;       /* E, CN_* info code */
    const double *dmin;        /* E, Danger.min_dist (inf when no human was closer) */
    const double *human_v;     /* 2 x H x E (component-major): cached ORCA velocities */
    const double *next_obs;    /* 5 x H x E (px py vx vy radius), update=0 only */
    const double *state;       /* 8 x (H+1) x E field-major SoA */
    const double *time;        /* E */
    const int32_t *action_idx; /* E, pending action index (-1 when set from raw xy) */
    const double *action_xy;   /* 2 x E pending action */
} cn_env_views;
int cn_env_get_views(cn_env *env, cn_env_views *out);

/* Blocking host read of (reward, done, info, dmin); any pointer may be NULL. */
int cn_env_read_outputs(cn_env *env, double *reward, uint8_t *done, uint8_t *info, double *dmin, void *stream);
/* Blocking host read of the ORCA velocities as E x H x 2 doubles. */
int cn_env_read_human_actions(cn_env *env, double *human_vxy_host, void *stream);
/* Blocking host read of update=0 observations as E x H x 5 doubles. */
int cn_env_read_next_obs(cn_env *env, double *obs_host, void *stream);
/* Blocking host read of the pending action: xy as E x 2 doubles and/or the action index (E int32, -1 when the
 * action did not come from the lookahead table); either pointer may be NULL. */
int cn_env_read_actions(cn_env *env, double *action_xy_host, int32_t *action_idx_host, void *stream);
/* Human velocities for the next cn_env_step from the HOST (E x H x 2 doubles) instead of an ORCA solve: the hook a learned
 * world model uses (ModelCrowdSim.step, model_crowd_sim.py:397-407,424-425: humans move with the velocities predicted by
 * sim_world).  Valid for one step, like the cached ORCA result it replaces. */
int cn_env_set_human_actions(cn_env *env, const double *human_vxy_host, void *stream);
/* Set the pending action from the host: E x 2 doubles. */
int cn_env_set_actions(cn_env *env, const double *action_xy_host, void *stream);
/* Blocking: reduce the device accumulators (explorer.py counters).  reset != 0 clears them. */
int cn_env_read_stats(cn_env *env, cn_stats *out, int reset, void *stream);
/* The per-ENV episode accumulators behind cn_env_read_stats, un-reduced: 11 arrays of E entries each, in this order --
 * int64 episodes, success, collision, timeout, steps, too_close; double sum_min_dist, sum_success_time,
 * sum_collision_time, sum_timeout_time, sum_return (table_host: cn_env_episode_table_bytes(env) bytes).  With auto_reset
 * off every env runs ONE episode and then freezes, so after a roll-out row e IS the outcome of episode e: this is how
 * Explorer.run_k_episodes (explorer.py:36-151) gets its per-episode results without a host sync per step.
 * frozen_host (optional, E bytes): 1 = the env's episode has ended.  Blocking. */
/* Outputs of the last cn_env_step copied device -> device into caller tensors (E doubles / E bytes each, any may be
 * NULL), asynchronously on `stream`: a roll-out that fills the replay memory records its per-step rewards and done flags
 * this way instead of reading them back (explorer.py:62-69,87-89).  A frozen env reports reward 0, done 1. */
int cn_env_copy_outputs(cn_env *env, double *reward_dev, uint8_t *done_dev, uint8_t *info_dev, void *stream);
int64_t cn_env_episode_table_bytes(const cn_env *env);
int cn_env_read_episode_table(cn_env *env, void *table_host, uint8_t *frozen_host, void *stream);

/* ---- policy: replaces policy_factory['sarl']() + configure (sarl.py:68-89) ---- */
int cn_policy_create(const cn_sarl_cfg *cfg, int device, cn_policy **out);
int cn_policy_destroy(cn_policy *p);
int64_t cn_policy_param_count(const cn_sarl_cfg *cfg);
/* model.load_state_dict (test.py:59): flat fp32 parameters in state-dict order
 * mlp1.{0,2} mlp2.{0,2} attention.{0,2,4} mlp3.{0,2,4,6}, each .weight ([out][in] row-major) then .bias.  attention.0.weight
 * is [attn_dims[0]][2 * mlp1_dims[1]] ([mlp1_out | group mean] columns), or [attn_dims[0]][mlp1_dims[1]] with
 * without_global_state. */
int cn_policy_load_weights(cn_policy *p, const float *flat_host, int64_t n, void *stream);
/* CADRL.build_action_space (cadrl.py:82-102), holonomic; out: A x 2 doubles; returns A via *n_actions. */
int cn_policy_action_table(cn_policy *p, double *out_xy_host, int32_t *n_actions);

/* MultiHumanRL.predict for every env (multi_human_rl.py:11-63): rotate, propagate the A actions,
 * reward + gamma_bar * V through mlp1 -> attention -> mlp3, first-strict-max argmax.
 * query_env != 0 uses the cached ORCA velocities and the env reward ladder (crowd_sim.py:325-329),
 * else constant-velocity humans and compute_reward (multi_human_rl.py:65-88).
 * epsilon > 0 applies the train-phase epsilon-greedy draw (multi_human_rl.py:28-30) from a per-env
 * Philox stream.  Writes the env's pending action. */
int cn_policy_lookahead(cn_policy *p, cn_env *env, int query_env, double epsilon, void *stream);
/* Blocking host read of the last lookahead: best_idx E int32, values E x A doubles (NULL to skip).
 * Returns CN_EVALUE when some env had no finite value (reference raises ValueError). */
int cn_policy_read(cn_policy *p, cn_env *env, int32_t *best_idx, double *values, void *stream);
/* Envs whose 81 action values were ALL non-finite since the handle was created (or since the last reset = 1 call): the
 * reference raises ValueError('Value network is not well trained.') for such a state (multi_human_rl.py:57-58).  The
 * blocking calls (cn_policy_read, cn_rollout_step_host, cn_rollout_step_host_packed) return CN_EVALUE themselves; the
 * device-resident and async forms (cn_rollout_step, _sharded, _host_packed_async) substitute action 0 and keep going, so
 * their callers poll this counter (blocking: one 4-byte D2H copy). */
int cn_policy_bad_count(cn_policy *p, int64_t *count, int reset, void *stream);

/* MultiHumanRL.transform (multi_human_rl.py:90-104) for every env: E x H x 13 fp32 into a DEVICE buffer. */
int cn_policy_transform(cn_policy *p, cn_env *env, float *out_dev, void *stream);
/* What predict() leaves in policy.last_state in the train phase (multi_human_rl.py:60-61): transform() of the state
 * predict() saw.  Identical to cn_policy_transform except for CN_NET_LSTM_RL, whose predict() first sorts the humans by
 * decreasing distance to the robot (lstm_rl.py:99-104), so the rows come out in that order. */
int cn_policy_last_state(cn_policy *p, cn_env *env, float *out_dev, void *stream);
/* ValueNetwork.forward (sarl.py:28-65) on a DEVICE batch x: B x H x 13 fp32 -> B fp32 (FP32 path;
 * used for TD targets, explorer.py:168-174). */
int cn_policy_forward(cn_policy *p, const float *x_dev, int32_t batch, int32_t human_num, float *out_dev,
                      void *stream);

/* ---- the fused hot path: one env step preceded by one full lookahead ---- */
/* orca -> lookahead -> step(update=1) [-> auto reset], all on `stream`, no host round trip.
 * This is what Explorer.run_k_episodes' inner loop (explorer.py:62-69) does per env. */
int cn_rollout_step(cn_policy *p, cn_env *env, int query_env, double epsilon, void *stream);
/* Same step for ONE SHARD of a batch that the caller has split into several env handles, each stepped on its own
 * stream (device-resident state, nothing synchronises): the kernels after the row kernel run on an internal
 * high-priority stream and `stream` is made to wait for them, so that one shard's feature / small kernels run beside
 * another shard's persistent row kernel instead of between two of them. */
int cn_rollout_step_sharded(cn_policy *p, cn_env *env, int query_env, double epsilon, void *stream);
/* ---- whole episodes: explorer.py:53-69 (`while not done: action = robot.act(ob); ob, reward, done, info = env.step(action)`)
 * for every env of the batch, enqueued natively: per step [transform -> record] humans (ORCA, or the world model of
 * ModelCrowdSim when `world` is given) -> robot action -> step(update=1) [-> record reward / done], no host round trip.  The env
 * must have auto_reset = 0: finished envs freeze, and every `check_every` steps the number of running envs is read back
 * asynchronously (looked at one interval later, so the stream never drains); the loop stops after max_steps or once that
 * count was zero.  *steps_run = steps enqueued (>= the longest episode).  Outcomes: cn_env_read_episode_table.
 * robot_mode: CN_ROBOT_POLICY = the lookahead of `p` (explorer.py:63 with a value-network policy), CN_ROBOT_ORCA = the
 * robot's own ORCA with `safety_space` (imitation learning, train.py:157-166), CN_ROBOT_KEEP = the pending action is kept
 * (run_k_episodes(stay=True) after cn_env_set_actions(0, 0)).
 * rec (optional) fills the replay-side records of explorer.py:60-69,87-89 as DEVICE arrays: states_dev[t] = what
 * transform_policy.transform (last_state = 0) / predict()'s last_state (1) gives for the state BEFORE step t
 * ((max_steps, E, H, input_dim) fp32), reward_dev[t], done_dev[t] ((max_steps, E) f64 / u8). */
enum { CN_ROBOT_POLICY = 0, CN_ROBOT_ORCA = 1, CN_ROBOT_KEEP = 2 };
typedef struct cn_world cn_world;
typedef struct cn_rollout_record {
    cn_policy *transform_policy;
    int32_t last_state;
    float *states_dev;
    double *reward_dev;
    uint8_t *done_dev;
} cn_rollout_record;
int cn_rollout_episodes(cn_policy *p, cn_env *env, cn_world *world, int robot_mode, double safety_space, int query_env,
                        double epsilon, int32_t max_steps, int32_t check_every, const cn_rollout_record *rec,
                        int32_t *steps_run, void *stream);
/* Same through HOST buffers (blocking): uploads agents/times (E x (H+1) x 8, E), runs the step and
 * downloads the new state, reward, done, info and the chosen action index.  Pinned memory recommended. */
int cn_rollout_step_host(cn_policy *p, cn_env *env, int query_env, double epsilon, const double *agents_in,
                         const double *times_in, double *agents_out, double *times_out, double *reward,
                         uint8_t *done, uint8_t *info, int32_t *action_idx, void *stream);

/* Same with ONE host->device and ONE device->host copy per step through packed blocks (pinned memory recommended):
 *   host_in : [agents E x (H+1) x 8 f64 | times E f64]                                      cn_host_step_bytes(env, 0)
 *   host_out: [agents | times | reward E f64 | action_idx E i32 | done E u8 | info E u8]      cn_host_step_bytes(env, 1)
 * The prefix of an output block is a valid input block, so a host loop can ping-pong two blocks without copying. */
int cn_rollout_step_host_packed(cn_policy *p, cn_env *env, int query_env, double epsilon, const void *host_in,
                                void *host_out, void *stream);
int64_t cn_host_step_bytes(const cn_env *env, int out);
/* Non-blocking form: enqueues copy-in, step and copy-out on `stream` and returns; host_out is valid after
 * cn_stream_sync(device, stream).  A host loop that owns several env shards (one stream, one policy handle and one
 * pair of pinned blocks per shard) overlaps the PCIe copies of one shard with the kernels of another: this is how a
 * host-resident driver of explorer.py:62-69 keeps the GPU busy.  Pinned host memory is REQUIRED for the overlap. */
int cn_rollout_step_host_packed_async(cn_policy *p, cn_env *env, int query_env, double epsilon, const void *host_in,
                                      void *host_out, void *stream);
int cn_stream_sync(int device, void *stream);

/* Developer diagnostic: timeline of the library's stream operations (named CUDA events).  cn_debug_trace(1) starts a
 * fresh recording, cn_debug_trace(0) stops; cn_debug_trace_dump synchronises and writes "ms stream name" lines. */
int cn_debug_trace(int on);
int cn_debug_trace_dump(char *buf, int64_t cap);

/* Number of kernels this library launched so far in this process. */
int64_t cn_launch_count(void);

/* Self-test of the tcgen05/TMEM building block: D[128 x N] = A[128 x K] * B[N x K]^T with fp16 operands,
 * fp32 accumulate.  a_host: 128 x K, b_host: N x K (row-major fp32, rounded to fp16 inside), d_host: 128 x N. */
int cn_selftest_umma(int32_t N, int32_t K, const float *a_host, const float *b_host, float *d_host, int device);
/* Same product with the B operand read MN-major from an activation-style image (rows = K index, K <= 128):
 * the form the kernel uses to sum the attention-weighted features over the humans of a group. */
int cn_selftest_umma_bmn(int32_t N, int32_t K, const float *a_host, const float *b_host, float *d_host, int device);
/* Same product with the A operand read from TMEM (packed fp16, "TS" mode): the form in which an activation that was
 * packed in place by an epilogue feeds the next layer without touching shared memory. */
int cn_selftest_umma_ts(int32_t N, int32_t K, const float *a_host, const float *b_host, float *d_host, int device);

/* CTA-pair building block (tcgen05 cta_group::2, M = 256 over the two SMs of a cluster, B split in N halves):
 * D[256 x N] = A[256 x K] * B[N x K]^T, repeated `reps` times; *cycles (optional) = clock64() ticks of the loop. */
int cn_selftest_umma_pair(int32_t N, int32_t K, const float *a_host, const float *b_host, float *d_host, int32_t reps,
                          long long *cycles, int device);

/* Developer diagnostic: clock64() at the phase boundaries of one tile of the tensor-core row kernel (CTA 0).
 * The first call arms the probes; call again after a lookahead to read 16 timestamps. */
int cn_debug_tc_timing(cn_policy *p, long long *out16);
/* CrowdSim.reset's scene generator on the host (crowd_sim.py:165-217,261-323), bit-identical to the reference: case i is
 * drawn from numpy's legacy MT19937 stream seeded with seeds[i] (= counter_offset[phase] + case id, crowd_sim.py:282-286).
 * rule = CN_CIRCLE_CROSSING / CN_SQUARE_CROSSING; agents_out: n x (human_num + 1) x 8 doubles in the exchange layout of
 * cn_env_set_state.  Host-only, multi-threaded; no device work. */
int cn_scenes_generate(int32_t n, const int64_t *seeds, int32_t human_num, int32_t rule, double circle_radius,
                       double square_width, double human_radius, double human_v_pref, double discomfort_dist,
                       double robot_radius, double robot_v_pref, int32_t randomize_attributes, double *agents_out);

/* ---- learned human-motion models of ModelCrowdSim (crowd_nav/policy/world_model.py:20-106, model_crowd_sim.py:397-425) ----
 * cn_world_create: CN_WORLD_ATTENTION (AttentionWorld, any human count <= 32) or CN_WORLD_MLP (MlpWorld(human_num)).
 * cn_world_load_weights: flat fp32 HOST array in the torch state-dict order of the reference module (its checkpoints load
 *   unchanged: mlp1.0 ... mlp3.6 / mlp.0, mlp.3, mlp.6, mlp.8; weight [out][in], then bias).
 * cn_world_predict: every human's next velocity from the env's CURRENT human states (px, py, vx, vy as fp32, like the
 *   reference's torch.Tensor([...])), written where cn_env_orca puts the ORCA velocities: the following cn_env_step /
 *   cn_policy_lookahead(query_env) / cn_rollout_step consume it.  No host round trip. */
int cn_world_create(int32_t kind, int32_t human_num, int device, cn_world **out);
int cn_world_destroy(cn_world *w);
int64_t cn_world_param_count(const cn_world *w);
int cn_world_load_weights(cn_world *w, const float *flat_host, int64_t n, void *stream);
int cn_world_predict(cn_world *w, cn_env *env, void *stream);

/* ---- value-network training step on the device (crowd_nav/utils/trainer.py:36-82) ------------------------------------
 * One optimisation step of the reference Trainer -- zero_grad, model(inputs), MSELoss, backward, SGD(momentum).step -- as
 * two kernels on ONE flat fp32 parameter block in torch state-dict order (the block cn_policy_load_weights takes, the same
 * layer list; cn_trainer_param_count = cn_policy_param_count of the config; the torch model's parameters may be views of
 * it).  Networks covered (cn_sarl_cfg.network):
 *   CN_NET_SARL      SARL with or without the global state (without_global_state); with_om = 1: OM-SARL, mlp1.0 reads
 *                    input_dim = 13 + cell_num^2 * om_channel_size columns (CN_EINVAL when input_dim disagrees).
 *   CN_NET_CADRL     value_network = mlp(13 -> mlp3_dims) on single-human states (cadrl.py:209): max_humans and human_num
 *                    must be 1 (CN_EINVAL otherwise); the batch is batch x input_dim.
 *   CN_NET_LSTM_RL   ValueNetwork1 (lstm_mlp1_dims[0] == 0): nn.LSTM(input_dim -> lstm_hidden) over the human_num rows in the
 *                    given order, then mlp(self_state_dim + lstm_hidden -> mlp3_dims) on [state[:, 0, :self_state_dim] | h_n];
 *                    ValueNetwork2 (lstm_mlp1_dims[0] > 0): a per-row mlp1 in front of the LSTM.  With or without maps.
 *                    Layout [mlp1.*] mlp.* lstm.weight_ih_l0, weight_hh_l0, bias_ih_l0, bias_hh_l0 (gates i, f, g, o).
 * Limits: 1 <= max_humans <= 16 (SARL: CN_EINVAL above; CADRL and LSTM-RL: CN_EUNSUPPORTED); shapes whose activations and
 * largest weight block (LSTM-RL: weight_hh, 4 lstm_hidden^2 floats) do not fit one CTA's shared memory: CN_EUNSUPPORTED.
 * cn_trainer_step: states_dev batch x human_num x input_dim fp32, targets_dev batch fp32 (device pointers).
 *   grad_out_dev == NULL : w_dev is updated in place (buf = momentum * buf + grad; w -= lr * buf), loss_dev (optional)
 *                          receives the batch MSE.
 *   grad_out_dev != NULL : only the gradient of the batch MSE is written (n_params fp32); the caller all-reduces it over
 *                          the ranks (NCCL) and calls cn_trainer_apply(grad, 1 / world) -- the data-parallel step.
 * cn_trainer_sync_weights: call after w_dev was changed by anyone else (load_state_dict, broadcast): refreshes the
 *   transposed copy the forward pass reads; zero_momentum = 1 also resets the momentum buffer (a new optimiser). */
typedef struct cn_trainer cn_trainer;
int cn_trainer_create(const cn_sarl_cfg *cfg, int device, int32_t max_batch, int32_t max_humans, cn_trainer **out);
int cn_trainer_destroy(cn_trainer *t);
int64_t cn_trainer_param_count(const cn_trainer *t);
int cn_trainer_sync_weights(cn_trainer *t, const float *w_dev, int zero_momentum, void *stream);
int cn_trainer_step(cn_trainer *t, float *w_dev, const float *states_dev, const float *targets_dev, int32_t batch,
                    int32_t human_num, float lr, float momentum, float *grad_out_dev, float *loss_dev, void *stream);
/* The same step with the batch GATHERED inside the kernel: sample i = item index_dev[i] (int64, device) of the replay
 * tensors memory_states_dev (capacity x human_num x input_dim fp32) / memory_values_dev (capacity fp32) -- what
 * DataLoader + collate_fn do on the host in the reference (trainer.py:9-17,68).  loss_sum_dev (optional) is ADDED to, so a
 * whole optimize_batch call reads the loss back once. */
int cn_trainer_step_indexed(cn_trainer *t, float *w_dev, const float *memory_states_dev, const float *memory_values_dev,
                            const int64_t *index_dev, int32_t batch, int32_t human_num, float lr, float momentum,
                            float *grad_out_dev, float *loss_sum_dev, void *stream);
int cn_trainer_apply(cn_trainer *t, float *w_dev, const float *grad_dev, float grad_scale, float lr, float momentum,
                     void *stream);

/* Measurement hook (bench.py `roofline`): on = 1 makes every later tensor-core lookahead record CUDA events around its
 * four kernels on the launching stream; out4 (optional) = durations of the LAST lookahead in ms {tc_features_kernel,
 * tc_rows_pair_kernel, tc_mlp3_pair_kernel, argmax_kernel} (blocks on the last event). */
int cn_debug_kernel_ms(cn_policy *p, int on, float *out4);

#ifdef __cplusplus
}
#endif
#endif

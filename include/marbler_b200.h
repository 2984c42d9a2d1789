/* marbler_b200 -- C ABI of the batched MARBLER environment step on B200 (sm_100a).
 *
 * The reference (GT-STAR-Lab/MARBLER) is pure Python and has NO FFI of its own for this path; the
 * only native boundary it crosses is cvxopt's CPython extension (SURVEY.md 8b).  The entry points
 * below are therefore the binding surface a maintainer would add (INTEGRATION.md shows the ctypes
 * stub); each cites the reference interface it replaces.  Conventions: extern "C", plain pointers
 * and sizes, no C++/torch types, no exceptions; 0 = ok, <0 = error (text via mrb_last_error).
 * Stream-ordered: every call enqueues on the caller's CUDA stream and (except *_host) never
 * synchronises.  The library never allocates caller-visible buffers: state / output buffers are
 * device memory owned by the caller (PyTorch tensors) and handed over with mrb_bind.
 * One handle per (process, GPU); a handle is not thread-safe (the reference is single-threaded).
 */
#ifndef MARBLER_B200_H
#define MARBLER_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define MRB_ABI_VERSION 7
#define MRB_MAX_ROBOTS 32
#define MRB_MAX_PREY 32

/* scenario ids: robotarium_gym/wrapper.py:12-16 env_dict, robotarium_gym/__init__.py:4-10 */
enum { MRB_PCP = 0, MRB_WAREHOUSE = 1, MRB_MATERIAL = 2, MRB_ARCTIC = 3, MRB_SIMPLE = 4 };
/* message codes: roboEnv.py:85-90 '' / 'collision' / 'boundary' / 'collision_boundary' */
enum { MRB_MSG_NONE = 0, MRB_MSG_COLLISION = 1, MRB_MSG_BOUNDARY = 2, MRB_MSG_COLLISION_BOUNDARY = 3 };
enum { MRB_OK = 0, MRB_E_ARG = -1, MRB_E_CUDA = -2, MRB_E_UNSUPPORTED = -3, MRB_E_STATE = -4 };

/* grid spawn sampler = rps generate_initial_conditions + utilities/misc.py:49-63
 * generate_initial_locations:  x = ((ix*spacing - w2) + sx1) + sx2,  y = ((iy*spacing - h2) + sy1) + sy2,
 * (ix, iy) = divmod(cell, yr), `count` distinct cells of the xr*yr grid. */
typedef struct mrb_spawn {
    int32_t count, xr, yr, random_theta;
    double spacing, w2, h2, sx1, sx2, sy1, sy2;
} mrb_spawn;

/* The scenario config.yaml keys the step path reads (SURVEY.md Appendix B), already resolved. */
typedef struct mrb_config {
    int32_t struct_size;            /* sizeof(mrb_config), checked by mrb_create */
    int32_t scenario;               /* MRB_PCP ... */
    int32_t num_robots;             /* PCP: predator+capture (PredatorCapturePrey.py:19); else n_agents; 2..32 */
    int32_t update_frequency;       /* roboEnv.py:52 */
    int32_t ctrl_period;            /* 15, roboEnv.py:63 */
    int32_t robotarium;             /* roboEnv.py:63: controller every sub-step */
    int32_t penalize_violations;    /* roboEnv.py:82 */
    int32_t barrier_default;        /* 0 'safe' (certificate2, r=.2), 1 'default' (r=.17): controller.py:13-16 */
    int32_t max_episode_steps;
    int32_t num_neighbors;          /* PCP / Warehouse */
    int32_t capability_aware;       /* PCP / MaterialTransport */
    int32_t num_prey, num_predators;                 /* PCP */
    int32_t n_fast, small_torque, large_torque;      /* MaterialTransport */
    int32_t auto_reset;             /* re-sample finished envs at the end of mrb_step */
    int32_t track_dist;             /* info['dist_travelled'] (roboEnv.py:55-56,93) */
    int32_t collect_stats;          /* episode statistics vector, see mrb_buffers.stats */
    int32_t reserved0;
    double left, right, up, down;   /* LEFT/RIGHT/UP/DOWN */
    double step_dist;               /* step_dist; ArcticTransport normal_step */
    double fast_step, slow_step;    /* MaterialTransport / ArcticTransport */
    double predator_radius, capture_radius;
    double time_penalty, sense_reward, capture_reward;
    double load_reward, unload_reward, goal_width;   /* Warehouse; MT: load/unload multiplier, end_goal_width */
    double zone1_radius;
    double not_reached_penalty, dist_multiplier;     /* ArcticTransport */
    double reward_scaler;                            /* Simple */
    double violation_reward;        /* -5 / -5 / -6 / -30 / -5 (literals in each scenario's step()) */
    double zone_mu[2], zone_sigma[2];                /* MaterialTransport zone1/zone2 normal(loc, scale) */
    mrb_spawn spawn_robots, spawn_other;             /* robots; PCP prey / Simple goal */
    /* rps RobotariumABC._validate collision test (roboEnv.py:80-94 reads its counters): a pair collides when
     * |(p_j + collision_offset (cos th_j, sin th_j)) - (p_k + collision_offset (cos th_k, sin th_k))| <= collision_diameter.
     * rps is not vendored in the reference and its pinned commit (6bb184e) cannot be read in the build container,
     * so both published forms are supported: centre to centre (collision_offset = 0; the SURVEY.md App. A.4
     * restatement, the default of the Python layer) and heading-projected points (collision_offset = 0.025). */
    double collision_diameter, collision_offset;
} mrb_config;

/* Caller-owned device buffers.  State is structure-of-arrays with the env index fastest:
 *   state_f64[row][env], state_i32[row][env]   (row counts from mrb_state_rows; rows named in
 *   marbler_b200/layout.py and DESIGN.md).  Outputs:
 *   obs f32 [B][N][D] | reward f32 [B][N] | done u8 [B] | message u8 [B] | remaining i32 [B] |
 *   dist f32 [B][N] (may be NULL when track_dist == 0) | stats f64 [MRB_NUM_STATS] (may be NULL). */
#define MRB_NUM_STATS 16
enum { MRB_STAT_EPISODES = 0, MRB_STAT_RETURN = 1, MRB_STAT_LENGTH = 2, MRB_STAT_COLLISION = 3,
       MRB_STAT_BOUNDARY = 4, MRB_STAT_SCENARIO = 5, MRB_STAT_ENV_STEPS = 6, MRB_STAT_QP_SOLVES = 7,
       MRB_STAT_QP_ITERS = 8, MRB_STAT_TIMEOUTS = 9,
       MRB_STAT_QP_STALLS = 10, /* solves that ran >= 25 iterations: cvxopt's iteration caught in a limit cycle */
       MRB_STAT_SUBSTEPS = 11,  /* simulator sub-steps executed (update_frequency per env step unless a violation ends it early) */
       /* iterations the hardware ran for the solves: with one env per thread a warp iterates until its slowest
        * env has converged, so this is the sum over solves of (warp maximum x lanes of the warp); divided by
        * MRB_STAT_QP_ITERS it is the divergence overhead of the solver loop (1.0 for the one-env-per-warp kernels) */
       MRB_STAT_QP_ITERS_WARP = 12 };
typedef struct mrb_buffers {
    double *state_f64;
    int32_t *state_i32;
    float *obs;
    float *reward;
    uint8_t *done;
    uint8_t *message;
    int32_t *remaining;
    float *dist;
    double *stats;
    /* optional float64 copies of obs / reward (NULL = off).  The reference returns float64 numpy observations and
     * Python-float rewards (e.g. PredatorCapturePrey.py:176); the single-env drop-in path binds these so that its
     * return values are not rounded through float32. */
    double *obs_f64;    /* [B][N][D] */
    double *reward_f64; /* [B][N] */
} mrb_buffers;

typedef struct mrb_env mrb_env;

int mrb_version(void);
/* replaces Wrapper.__init__ -> env_dict[env_name](args) (wrapper.py:20-34): builds the handle for
 * num_envs independent envs whose global ids are env_id0 .. env_id0+num_envs-1 (RNG stream offset
 * of this rank when envs are sharded over GPUs). */
int mrb_create(const mrb_config *cfg, int device, int64_t num_envs, int64_t env_id0, mrb_env **out);
int mrb_destroy(mrb_env *env);
const char *mrb_last_error(const mrb_env *env);          /* env may be NULL: last create error */
/* layout queries (spaces: <Scenario>.get_observation_space / get_action_space) */
int mrb_state_rows(const mrb_env *env, int32_t *rows_f64, int32_t *rows_i32);
int mrb_obs_dim(const mrb_env *env);
int mrb_num_actions(const mrb_env *env);
int mrb_bind(mrb_env *env, const mrb_buffers *buffers);
/* replaces <Scenario>.reset() + roboEnv.reset() (e.g. PredatorCapturePrey.py:114-136,
 * roboEnv.py:27-36,98-118).  mask: device u8[B] (NULL = all envs).  Zeroes obs of the reset envs
 * (the reference returns an all-zero observation from reset). */
int mrb_reset(mrb_env *env, const uint8_t *mask, uint64_t seed, void *cuda_stream);
/* replaces Wrapper.step(action_n) (wrapper.py:41-44) -> <Scenario>.step -> roboEnv.step
 * (roboEnv.py:38-96) -> Controller.set_velocities (controller.py:20-25) -> rps / cvxopt.
 * actions: device i32 [B][N]. */
int mrb_step(mrb_env *env, const int32_t *actions, void *cuda_stream);
/* ---- masked step (EPyMARL's ParallelRunner steps only envs_not_terminated and leaves the others alone until the batch
 * ends).  active: device u8 [B] on the env's device; an env b with active[b] != 0 is stepped exactly as mrb_step steps
 * it - its state and every output row (obs, reward, done, message, remaining, dist, obs_f64, reward_f64) bit for bit,
 * auto-reset included.  Of an env with active[b] == 0 nothing is read or written: no state row, no output row, no
 * auto-reset, no contribution to stats.  The integer stats counters (env steps, QP solves and iterations, sub-steps,
 * episodes, collisions, boundary exits, timeouts) count exactly the active env-steps; the float sums (return, length)
 * are those of the same episodes up to the order of the atomic additions.  active == NULL is mrb_step.
 * Two launches whatever the mask holds: a compaction of `active` into a list of active env ids (library-internal
 * scratch allocated by mrb_create), then the step kernel over that list with its grid sized for B, so a captured CUDA
 * graph keeps its shape.  Stream-ordered, never synchronises, capturable; the caller keeps `active` unchanged until
 * the launches have run.  Every argument is checked before the device is touched: as mrb_step, plus an `active` that is
 * not device memory of the env's device (cudaPointerGetAttributes) -> MRB_E_ARG.  mrb_step_host has no mask. */
int mrb_step_masked(mrb_env *env, const int32_t *actions, const uint8_t *active, void *cuda_stream);
/* same step with HOST buffers (pinned for full speed; pageable works): H2D actions, step, D2H
 * obs/reward/done/message, then synchronises.  Batches of >= 16,384 envs are cut into up to 8 chunks,
 * each on its own library-internal stream (ordered after the caller's stream), so that the PCIe copies
 * of one chunk overlap the kernels of the others.  NULL host outputs are skipped.  When every buffer
 * is pinned (cudaHostAlloc / cudaHostRegister) the kernel stores reward / done / message directly into
 * the host buffers through their device aliases and only obs is downloaded by the copy engine;
 * environment MRB_HOST_DIRECT=1 sends obs the same way, =0 downloads everything.  The device-side
 * buffers bound with mrb_bind are written in every mode. */
int mrb_step_host(mrb_env *env, const int32_t *actions_host, float *obs_host, float *reward_host,
                  uint8_t *done_host, uint8_t *message_host, void *cuda_stream);
/* ---- state access by field (checkpoint / restore, parity injection).  The reference keeps this state in Python
 * attributes of the scenario, its agents and roboEnv (cited per field); here it is packed into the SoA rows of
 * state_f64 / state_i32, and these two calls convert between the rows and plain per-field HOST arrays for the envs
 * [env_lo, env_lo + count).  NULL fields are skipped (get) / left unchanged (set); fields of other scenarios are
 * ignored.  Both calls are ordered after the work already enqueued on cuda_stream and synchronise before returning. */
typedef struct mrb_state_fields {
    int32_t struct_size;         /* sizeof(mrb_state_fields) */
    int32_t reserved0;
    double *poses;               /* [count][3][N]  scenario.agent_poses = robotarium.poses (x row, y row, theta row) */
    double *prev_pose;           /* [count][3][N]  roboEnv.previous_pose (roboEnv.py:55-59); only x, y are state, theta reads 0 */
    double *episode_return;      /* [count]        sum of team rewards of the running episode (statistics only) */
    int32_t *episode_steps;      /* [count]        scenario.episode_steps */
    int32_t *prev_valid;         /* [count]        roboEnv.previous_pose is not None (roboEnv.py:117) */
    int32_t *episode_count;      /* [count]        episodes started so far: Philox counter of the next auto-reset */
    double *prey_loc;            /* [count][P][2]  PCP prey_loc (PredatorCapturePrey.py:128-132) */
    uint8_t *prey_sensed;        /* [count][P]     PCP prey_sensed */
    uint8_t *prey_captured;      /* [count][P]     PCP prey_captured */
    uint8_t *loaded;             /* [count][N]     Warehouse agent.loaded (warehouse.py:145-178) */
    int32_t *load;               /* [count][N]     MaterialTransport agent.load */
    int32_t *zone_load;          /* [count][2]     MaterialTransport zone1_load, zone2_load (MaterialTransport.py:99-100) */
    int32_t *messages;           /* [count][4]     MaterialTransport messages (MaterialTransport.py:119-120) */
    uint8_t *grid;               /* [count][8][12] ArcticTransport grid (ArcticTransport.py:56-82) */
    int32_t *goal_col;           /* [count]        ArcticTransport goal_loc[1] */
    int32_t *pixel_type;         /* [count][N]     ArcticTransport agent.pixel_type (agent.py:37-39) */
    uint8_t *reached_goal;       /* [count][N]     ArcticTransport agent.reached_goal */
    double *goal;                /* [count][2]     Simple goal_loc (simple.py:141-144) */
} mrb_state_fields;
int mrb_get_state(mrb_env *env, int64_t env_lo, int64_t count, const mrb_state_fields *out, void *cuda_stream);
int mrb_set_state(mrb_env *env, int64_t env_lo, int64_t count, const mrb_state_fields *in, void *cuda_stream);

/* unit entry for the barrier-certificate QP alone (rps create_single_integrator_barrier_certificate{,2}
 * -> cvxopt.solvers.qp; called at controller.py:23).  Device SoA: dxi, xi, u are f64 [2][N][B];
 * iters i32 [B] (may be NULL). */
int mrb_barrier_qp(int device, int32_t num_robots, int32_t barrier_default, int64_t num_problems,
                   const double *dxi, const double *xi, double *u, int32_t *iters, void *cuda_stream);

/* ---- on-device policy (SURVEY.md section 8f-1): the reference's evaluation loop utilities/misc.py:134-221
 * (run_env) calls utilities/rnn_agent.py:5-29 RNNAgent / utilities/rnn_ns_agent.py:5-36 RNNNSAgent on the
 * host once per env step: q, h = model(obs, h); actions = argmax(q).  mrb_policy_act does that for every
 * agent of every env in one kernel: fc1 -> ReLU -> GRUCell (or Linear+ReLU when use_rnn == 0) -> fc2 ->
 * greedy argmax, tensor-core MMAs on FP16 operands with FP32 accumulation and FP32 gates (tcgen05 / TMEM for
 * hidden 128 + GRUCell with <= 8 actions, mma.sync otherwise) - or, with desc.accurate, in float32 throughout -,
 * reading the env's obs buffer and writing the actions buffer mrb_step consumes (no host round trip). */
typedef struct mrb_policy_desc {
    int32_t struct_size;        /* sizeof(mrb_policy_desc): ABI check */
    int32_t obs_dim;            /* D: width of one agent's row in the obs buffer */
    int32_t input_dim;          /* fc1.in_features = D (+ n_agents when obs_agent_id, misc.py:161-162) */
    int32_t hidden_dim;         /* 64 or 128 (model json "hidden_dim") */
    int32_t n_actions;          /* <= 24 */
    int32_t n_agents;
    int32_t obs_agent_id;       /* append the one-hot agent id to the observation */
    int32_t use_rnn;            /* 1: nn.GRUCell, 0: nn.Linear + ReLU (rnn_agent.py:11-14) */
    int32_t non_shared;         /* 1: one weight set per agent (RNNNSAgent), 0: one shared set */
    int32_t accurate;           /* 1: float32 operands and accumulation like the reference (plain FMA kernel, ~10x the
                                 * time): the greedy actions of a checkpoint are the reference's; 0: FP16 tensor-core
                                 * operands (q within ~1e-3 |q|, about one near-tie decision in a thousand differs) */
} mrb_policy_desc;
typedef struct mrb_policy mrb_policy;
/* weights: HOST float32, (non_shared ? n_agents : 1) sets back to back, each set in state_dict order and
 * torch layout ([out][in] row-major): fc1.weight, fc1.bias, then rnn.weight_ih [3H][H], rnn.weight_hh [3H][H],
 * rnn.bias_ih, rnn.bias_hh (use_rnn) or rnn.weight [H][H], rnn.bias (otherwise), then fc2.weight, fc2.bias.
 * Synchronous: uploads the weights to a temporary device buffer and builds the policy's images from it with the
 * kernel mrb_policy_load launches, on the legacy default stream. */
int mrb_policy_create(const mrb_policy_desc *desc, int device, const float *weights, int64_t num_weights,
                      mrb_policy **out);
/* Replace the weights of `policy` in place (EPyMARL's mac.load_state: the collecting policy follows the learner).
 * weights: DEVICE float32 on the policy's device, num_weights = the count mrb_policy_create took, same order.  Rebuilds
 * every image the policy holds on cuda_stream: one launch, no allocation, no host copy, no synchronisation; capturable
 * in a CUDA graph.  Graphs that captured mrb_policy_act on this policy stay valid and see the new weights at their next
 * replay.  Ordered after the work already on cuda_stream; the caller orders other streams (e.g. a learner's) before it,
 * and keeps `weights` unchanged until the launch has run.  Every argument is checked before the device is touched: a
 * NULL policy or weights, another count, weights that are not 4-byte aligned or not device memory of the policy's
 * device (cudaPointerGetAttributes) -> MRB_E_ARG, and the policy's images are untouched. */
int mrb_policy_load(mrb_policy *policy, const float *weights, int64_t num_weights, void *cuda_stream);
int mrb_policy_destroy(mrb_policy *policy);
const char *mrb_policy_last_error(const mrb_policy *policy);
/* obs f32 [B][N][D], hidden f32 [B][N][H] (in/out), actions i32 [B][N] (out), q f32 [B][N][n_actions] (out,
 * may be NULL), fresh u8 [B] (may be NULL): envs flagged != 0 start a new episode - their hidden state and
 * observation are taken as zero (run_env re-zeroes hs and feeds reset()'s all-zero obs, misc.py:156,219).
 * All device pointers; stream-ordered, no synchronisation.  hidden must be 16-byte aligned (MRB_E_ARG otherwise):
 * the kernels access it as float4; a contiguous view that starts a multiple of 4 floats into an allocation is. */
int mrb_policy_act(mrb_policy *policy, int64_t num_envs, const float *obs, float *hidden, int32_t *actions,
                   float *q, const uint8_t *fresh, void *cuda_stream);

/* ---- exploratory action selection (training-time data collection).  EPyMARL, which trains the reference's
 * checkpoints, does not act greedily while it collects data: QMIX / VDN / IQL use EpsilonGreedyActionSelector with a
 * linear DecayThenFlatSchedule, MAPPO / IPPO use SoftPoliciesSelector.  mrb_select_actions restates both over the
 * output of mrb_policy_act, one thread per (env, agent) row.
 *   MRB_SELECT_EPSILON_GREEDY: actions (in/out) holds the greedy actions on entry (q is not read and may be NULL);
 *     eps(t) = max(eps_finish, eps_start - (eps_start - eps_finish) * t / anneal_time) in double; a row explores iff
 *     w0 < (eps >= 1 ? 2^32 : floor(eps * 2^32)), and then takes action (w1 * n_actions) >> 32.
 *   MRB_SELECT_SOFTMAX: q f32 [B][N][n_actions] (in), actions (out): u = ((w2 >> 5) * 2^26 + (w3 >> 6)) / 2^53;
 *     in double, e_a = exp(q_a - max q), S = sum of e_a in index order; the action is the first a whose running sum
 *     exceeds u * S (the last a with e_a > 0 if rounding leaves none).
 * w0..w3 is one Philox4x32-10 block: key (seed lo, seed hi), counter (gid lo, gid hi, (uint32) t, 0x80000000 | agent),
 * gid = env_id0 + env.  t = *step, a device int64 that the call reads and then advances by one on the same stream
 * (a one-thread kernel after the selection kernel: two launches), so every replay of a captured CUDA graph moves the
 * schedule on.  The Philox counter takes t modulo 2^32: draws repeat after 2^32 steps of one counter. */
enum { MRB_SELECT_EPSILON_GREEDY = 1, MRB_SELECT_SOFTMAX = 2 };
typedef struct mrb_select_desc {
    int32_t struct_size;        /* sizeof(mrb_select_desc): ABI check */
    int32_t mode;               /* MRB_SELECT_* */
    uint64_t seed;
    int64_t env_id0;            /* global id of env 0 of this batch (sharding) */
    double eps_start, eps_finish;   /* epsilon-greedy: DecayThenFlatSchedule, linear; both in [0, 1] */
    int64_t anneal_time;        /* in steps of *step; >= 1 */
} mrb_select_desc;
/* errors through mrb_last_error(NULL); every argument is checked before the device is touched */
int mrb_select_actions(int device, int64_t num_envs, int32_t n_agents, int32_t n_actions,
                       const mrb_select_desc *desc, int64_t *step, const float *q, int32_t *actions,
                       void *cuda_stream);

/* ---- episode recording (training-time data collection).  EPyMARL's ParallelRunner.run fills an EpisodeBatch one
 * step at a time; mrb_record_begin / mrb_record_step write the same fields straight into caller-owned device tensors,
 * after every mrb_step, in one launch per step (EPyMARL is not vendored in the reference, so the contract is restated
 * here).  B envs (the env handle's), episode limit T (EPyMARL's time_limit), N agents, D = mrb_obs_dim, A =
 * mrb_num_actions, W = obs_width >= D (the declared observation width; columns D .. W-1 are zero, as the adapter's
 * padding).  Every field has T + 1 rows per env (max_seq_length = episode_limit + 1), all contiguous, row-major:
 *   obs f32 [B][T+1][N][W] | state f32 [B][T+1][N*W]: the same memory as obs (state = concat(obs)), state == obs |
 *   actions i64 [B][T+1][N] | actions_onehot f32 [B][T+1][N][A] | avail_actions i32 [B][T+1][N][A] |
 *   reward f32 [B][T+1] | terminated u8 [B][T+1] | filled i64 [B][T+1] | cursor i32 [B].
 * Every env records exactly one episode, starting at row 0 (ParallelRunner.reset):
 *   row 0: obs 0 (the reset observation), avail_actions 1, filled 1.
 *   step t (the t-th mrb_record_step since mrb_record_begin), for every env that has not terminated yet:
 *     actions[t] = the actions sent to the env (after exploration), actions_onehot[t] their one-hot encoding,
 *     reward[t] = the float32 sum of the N agent rewards in agent index order,
 *     terminated[t] = done || t + 1 >= T (truncation is stored as terminal: the gym wrapper reports no
 *     episode_limit info), obs[t+1] = the env's obs buffer after the step (the terminal observation of an env that
 *     has just finished), avail_actions[t+1] = 1, filled[t+1] = 1; the env is inactive from then on if terminated.
 *   every other element is 0, including actions, actions_onehot, reward and terminated of the terminal row and all
 *   the rows after it.
 * Each element is written exactly once per collection: mrb_record_begin writes row 0 of obs / avail_actions / filled
 * and row T of actions / actions_onehot / reward / terminated; step t writes row t of the latter four and row t + 1 of
 * the former three for every env, active or not (zeros for an inactive one), so after mrb_record_begin and T calls of
 * mrb_record_step every row has been written and the tensors need no zeroing.  cursor[b] is the recorder's position:
 * t while env b is active, ~t (= -t - 1) once it has terminated, t = the calls since mrb_record_begin; a call at
 * t >= T writes nothing.  Each env's cursor is read and written by that env's own thread of one launch.
 * Accesses are scalar and of the elements' own widths (no vector accesses): every pointer must be aligned to its
 * element size (8 bytes for actions and filled, 4 for the others), MRB_E_ARG otherwise. */
typedef struct mrb_episode_batch {
    int32_t struct_size;        /* sizeof(mrb_episode_batch): ABI check */
    int32_t episode_limit;      /* T: 1 .. 2^30 */
    int32_t obs_width;          /* W: D .. 65,536 */
    int32_t reserved0;
    float *obs;
    float *state;               /* == obs */
    int64_t *actions;
    float *actions_onehot;
    int32_t *avail_actions;
    float *reward;
    uint8_t *terminated;
    int64_t *filled;
    int32_t *cursor;
} mrb_episode_batch;
/* Brings the batch to its row-0 state (see above) and sets every cursor to 0.  One launch, stream-ordered.  Errors
 * through mrb_last_error(env) (mrb_last_error(NULL) when env is NULL); every argument is checked before the device is
 * touched: NULL pointers, struct_size, episode_limit, obs_width and alignment -> MRB_E_ARG, an env without buffers
 * (mrb_bind) -> MRB_E_STATE. */
int mrb_record_begin(mrb_env *env, const mrb_episode_batch *batch, void *cuda_stream);
/* Records the step that mrb_step just took with `actions` (device i32 [B][N], 4-byte aligned): reads the bound obs,
 * reward and done buffers.  One launch, stream-ordered, never synchronises; checks as mrb_record_begin. */
int mrb_record_step(mrb_env *env, const mrb_episode_batch *batch, const int32_t *actions, void *cuda_stream);

/* ---- evaluation (per-episode results, utilities/misc.py:134-221 run_env; EPyMARL's runner in test mode).
 * mrb_eval_step runs after every mrb_step and logs each env's first K finished episodes into a caller-owned table,
 * one launch per step.  It reads only the bound reward, done, message, remaining and (when bound) dist buffers.
 * B envs (the env handle's), N agents, all tensors contiguous, row-major, device memory:
 *   per episode [B][K]: return_ f64 | length i32 | message u8 | timeout u8 | remaining i32 | dist f32
 *   per env [B]: acc_return f64 | acc_length i32 | acc_dist f64 | count i32.
 * Every step, for every env: team = the float32 sum of the N agent rewards in agent index order, starting from 0
 * (the thread-per-env step kernels' episode return term; the team kernels of 7 or more robots sum with a warp
 * butterfly); acc_return += (double)team; acc_length += 1; acc_dist += the float64 sum, in agent index order starting
 * from 0, of the N floats of dist (0 when no dist buffer is bound).  Then, if done[b]:
 * when k = count[b] < K, row k gets return_ = acc_return, length = acc_length, message = the step's message (bit 0
 * collision, bit 1 boundary), timeout = (message == 0 && length > max_episode_steps, the MRB_STAT_TIMEOUTS test),
 * remaining = the step's remaining, dist = (float)acc_dist, and count[b] = k + 1; whether or not a row was written, the
 * three accumulators go back to 0.  An env with count == K logs nothing more.  Row k of env b is valid iff
 * k < count[b]; the table is never zeroed.  Each env's accumulators and count are read and written by that env's own
 * thread of one launch.  The lengths count steps since mrb_eval_begin, so call mrb_eval_begin together with mrb_reset
 * of every env (or at an episode boundary of every env).
 * Accesses are scalar and of the elements' own widths: every pointer must be aligned to its element size (8 bytes for
 * return_, acc_return and acc_dist, 4 for length, remaining, dist, acc_length and count), MRB_E_ARG otherwise. */
typedef struct mrb_eval_table {
    int32_t struct_size;        /* sizeof(mrb_eval_table): ABI check */
    int32_t episodes;           /* K: 1 .. 2^20 */
    double *return_;
    int32_t *length;
    uint8_t *message;
    uint8_t *timeout;
    int32_t *remaining;
    float *dist;
    double *acc_return;
    int32_t *acc_length;
    double *acc_dist;
    int32_t *count;
} mrb_eval_table;
/* Sets the accumulators and count of every env to 0 (the table rows are left as they are).  One launch,
 * stream-ordered, never synchronises, capturable.  Errors through mrb_last_error(env) (mrb_last_error(NULL) when env is
 * NULL); every argument is checked before the device is touched: NULL pointers, struct_size, episodes and alignment ->
 * MRB_E_ARG, an env without buffers (mrb_bind) -> MRB_E_STATE. */
int mrb_eval_begin(mrb_env *env, const mrb_eval_table *table, void *cuda_stream);
/* Logs the step that mrb_step just took (see above).  One launch, stream-ordered, never synchronises, capturable;
 * checks as mrb_eval_begin. */
int mrb_eval_step(mrb_env *env, const mrb_eval_table *table, void *cuda_stream);

/* FP64 roofline denominator, measured: runs a kernel of independent DFMA chains (8 per thread, one 1,024-thread
 * CTA per SM) for about `milliseconds` on `device`, timed with CUDA events, and returns the rate of the best launch
 * in TFLOP/s (2 flops per DFMA).  The env step is bound by FP64 issue, not by HBM (SURVEY.md 8d), so bench.py
 * reports the step kernels' FP64 flop rate against this number. */
int mrb_fp64_peak(int device, double milliseconds, double *tflops);

/* number of kernels this library has launched in the process so far (bench.py's gpu_launches) */
int64_t mrb_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif

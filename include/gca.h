/* gca.h - C ABI of libgca: the batched, device-resident step hot path of the
 * single-aircraft guidance / collision-avoidance environments, hand-written for sm_100a.
 *
 * The reference (xuxiyang1993/gym-guidance-collision-avoidance-single) is pure Python and has
 * no FFI of its own; each entry point below names the reference interface it replaces
 * (paths relative to the reference root, PKG = gym_guidance_collision_avoidance_single/envs).
 * INTEGRATION.md shows the ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *   - plain C, no torch / C++ types; every function returns 0 on success or a negative
 *     gca_status; the message for the calling thread's last failure is gca_last_error().
 *   - a gca_env handle is bound to one CUDA device and is not thread-safe.
 *   - entry points taking a `stream` (a cudaStream_t passed as void*) are asynchronous on that
 *     stream and never synchronise; the *_host entry points synchronise before returning.
 *   - device state is owned by the handle; input / output buffers are owned by the caller.
 *   - there is NO CPU implementation behind this ABI: without a usable CUDA device
 *     gca_create fails with GCA_ERR_CUDA.
 */
#ifndef GCA_H_
#define GCA_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GCA_ABI_VERSION 7

typedef enum gca_status {
  GCA_OK = 0,
  GCA_ERR_INVALID = -1, /* bad argument */
  GCA_ERR_CUDA = -2,    /* CUDA runtime error (message has the CUDA string) */
  GCA_ERR_ALLOC = -3,   /* host allocation failed */
  GCA_ERR_STATE = -4    /* call not valid in the handle's current configuration */
} gca_status;

/* numerics: FAITHFUL reproduces the reference's mixed f32/f64 arithmetic (SURVEY.md 8(a)
 * "Numerics contract"): f64-capable intruder positions, f64 observations and rewards.
 * FAST stores intruder positions in f32 only (a spawn that was retried is rounded to f32, the
 * one deviation from the reference, Q3) and emits f32 observations / rewards, i.e. exactly what
 * a baselines VecEnv hands to a learner (dummy_vec_env.py:25-27). */
enum { GCA_MODE_FAITHFUL = 0, GCA_MODE_FAST = 1 };

/* where random draws come from: TAPE replays values recorded from the reference's global
 * numpy stream in the reference's consumption order (per-env cursor); PHILOX generates them
 * on the device with Philox4x32-10 addressed by (seed; env id, tick, slot, block). */
enum { GCA_DRAWS_TAPE = 0, GCA_DRAWS_PHILOX = 1 };

/* action decoding (a2/a3/a3' in SURVEY.md 8(a)) */
enum {
  GCA_ACT_DISCRETE9 = 0,  /* int32 a: a0 = a / 3, a1 = a % 3, delta = (a0-1, a1-1)  PKG/SingleAircraftEnv.py:130-133,300-302;
                             also the (a0, a1) tuple of Simulators/SingleAircraftMCTSEnv.py:126-130 encoded a0*3+a1 */
  GCA_ACT_CONTINUOUS2 = 1, /* real a[2] in [-1,1]: delta = (a[0], a[1])              PKG/SingleAircraft2Env.py:292-294 */
  GCA_ACT_DISCRETE3 = 2,   /* int32 a: heading delta a-1, speed += speed_sigma       PKG/SingleAircraftDiscreteHEREnv.py:302-304 */
  GCA_ACT_DISCRETE3_HEADING = 3 /* int32 a: heading delta a-1, speed only clamped   Simulators/SingleAircraftDiscrete3HEREnv.py:407-411 */
};

/* observation layout (a9/a10/a16) */
enum {
  GCA_OBS_VECTOR = 0,   /* [intruders x4][own x6][goal x2], normalised   PKG/SingleAircraftEnv.py:100-126 */
  GCA_OBS_HER = 1,      /* [own x6][intruders x4] + achieved/desired normalised  PKG/SingleAircraftHEREnv.py:103-139 */
  GCA_OBS_DHER = 2,     /* as HER but achieved/desired are raw pixel positions   PKG/SingleAircraftDiscreteHEREnv.py:128-133 */
  GCA_OBS_RAW = 3,      /* VECTOR layout, un-normalised values     Simulators/SingleAircraftMCTSEnv.py:98-124 */
  GCA_OBS_NONE = 4,     /* no vector observation (StackEnv: the image comes from gca_raster) */
  GCA_OBS_NEAREST = 5,  /* [own x4][nearest_n intruders x5: x, y, vx, vy, dist / diagonal, nearest first] + achieved /
                           desired normalised; needs N > nearest_n
                           Simulators/SingleAircraftDiscrete9HEREnv.py:106-165 */
  GCA_OBS_RAW6 = 6      /* [intruders x6: x, y, vx, vy, speed, heading][own x6][goal x2], un-normalised
                           Simulators/SingleAircraftMCTSRandIntruderEnv.py:124-152 */
};

enum { GCA_WALL_NONE = 0, GCA_WALL_TERMINAL = 1, GCA_WALL_PENALTY = 2 };

/* per-step result code, the reference's info string ('' n c g w m) */
enum { GCA_INFO_NONE = 0, GCA_INFO_NMAC = 1, GCA_INFO_CONFLICT = 2, GCA_INFO_GOAL = 3, GCA_INFO_WALL = 4, GCA_INFO_MAXSTEPS = 5 };

/* Philox slot namespace: counter = (env id, tick, slot, block) */
#define GCA_SLOT_OWNSHIP 0x80000000u /* block 0: Box-Muller pair (heading noise, speed noise) */
#define GCA_SLOT_GOAL 0x40000000u    /* block 0: goal (x, y) of a reset */
#define GCA_SLOT_RESET 0x20000000u   /* | intruder index: spawn made by a reset */
#define GCA_SLOT_OWN_RESET 0x10000000u /* random_start: ownship drawn by a reset, blocks POS and SPEED_HEADING */
#define GCA_SLOT_TURN 0x08000000u    /* _update_headings: | pair index j, block 0 -> (p of intruder 2j, p of intruder 2j + 1);
                                        an intruder i with p < turn_prob takes u = first uniform of (| i, block 1) and
                                        turns by radians(-turn_max_deg + 2 * turn_max_deg * u) */
                                     /* intruder index alone: respawn made inside a step */
#define GCA_BLOCK_POS 0u             /* (x, y) */
#define GCA_BLOCK_SPEED_HEADING 1u   /* (speed, heading) */
#define GCA_BLOCK_RETRY0 2u          /* + r: r-th re-draw of (x, y) by the rejection loop */
#define GCA_MAX_SPAWN_RETRIES 64     /* PHILOX only: after this many rejections the position is accepted */

/* Parameters of one environment family.  Field names follow PKG/config.py:4-39 and
 * Simulators/config.py:4-55; the variant rows follow the reward table of SURVEY.md 8(a). */
typedef struct gca_config {
  double window_width, window_height;
  double minimum_separation, nmac_dist, initial_min_dist, goal_radius;
  double min_speed, max_speed, d_speed, speed_sigma;
  double d_heading, heading_sigma;
  /* values _get_ob re-reads from the Config class on every call (Q12) */
  double ob_window_width, ob_window_height, ob_min_speed, ob_max_speed;
  /* reward row */
  double r_nmac, r_conflict, r_wall, r_goal, r_default;
  int32_t shaped_default; /* 1: default reward is -dist(own, goal) / 1200; 0: r_default */
  int32_t action_kind;    /* GCA_ACT_* */
  int32_t obs_kind;       /* GCA_OBS_* */
  int32_t wall_kind;      /* GCA_WALL_* */
  int32_t max_steps;      /* > 0: StackEnv rule - steps >= max_steps ends the episode before intruders move */
  int32_t time_limit;     /* > 0: gym TimeLimit of the registered ids (timestep_limit=10000,
                             gym_guidance_collision_avoidance_single/__init__.py:9): after the step,
                             ep_steps >= time_limit also ends the episode (reward/info unchanged) */
  int32_t random_start;   /* 1: reset() draws the ownship - random_pos(), random_speed(), random_heading(), in that
                             order, before the intruders (Simulators/SingleAircraftDiscrete9HEREnv.py:78-82);
                             0: (50, 50), min_speed, pi/4 (PKG/SingleAircraftEnv.py:72-76) */
  int32_t nearest_n;      /* GCA_OBS_NEAREST: Config.n (Simulators/config.py:55), 1..8 */
  double ob_diagonal;     /* GCA_OBS_NEAREST: Config.diagonal, normalises the distance entry (Simulators/config.py:8) */
  /* Simulators/SingleAircraftDiscrete3HEREnv.py */
  double conflict_coeff;  /* shaped_nearest: r = conflict_coeff * dist_nearest_intruder - 0.1 when that distance is below
                             3 * minimum_separation, added to the default reward (:225-232; Simulators/config.py:44) */
  double goal_margin;     /* > 0: the goal is drawn in [margin, window - margin]^2 (random_goal_pos :349-353) */
  int32_t shaped_nearest; /* 1: track dist_nearest_intruder over the intruders the loop visited (:185,:191) */
  /* Simulators/SingleAircraftMCTSRandIntruderEnv.py */
  int32_t intruder_turns; /* 1: after _terminal_reward every intruder draws p = uniform() and, when p < turn_prob, turns by
                             radians(uniform(-turn_max_deg, turn_max_deg)): heading += delta, velocity = f32(speed * (cos,
                             sin)) (_update_headings :166-174, change_heading :332-336); needs per-intruder (heading,
                             speed) state */
  double position_drift;  /* added to both velocity components of every intruder advance, in f32:
                             position += velocity + Config.position_sigma (:183 - a constant, not a draw) */
  double turn_prob;       /* 0.1 (:170) */
  double turn_max_deg;    /* 10 (:173) */
} gca_config;

/* Canonical host-side view of the full simulator state, identical for both modes
 * (used by gca_get_state / gca_set_state and by the oracle).  Arrays are C-contiguous. */
typedef struct gca_host_state {
  float* own_pos;            /* [B][2]   f32 position            PKG/SingleAircraftEnv.py:271 */
  double* own_hs;            /* [B][2]   heading, speed          :272-273 */
  double* own_vel;           /* [B][2]   velocity :276,:308 */
  uint8_t* own_vel_is_f32;   /* [B]      velocity is still the f32 array made by reset (Q2) */
  double* goal;              /* [B][2]   :93 */
  int32_t* no_conflict;      /* [B]      :96 */
  int32_t* ep_steps;         /* [B]      steps since reset (StackEnv :118; TimeLimit) */
  uint32_t* tick;            /* [B]      Philox tick: +1 per step and per explicit reset of that env */
  double* ipos;              /* [B][N][2] intruder positions (f32-valued unless flagged) */
  uint8_t* ipos_is_f64;      /* [B][N]   position dtype is f64 (retried spawn, Q3) */
  float* ivel;               /* [B][N][2] :276 */
  uint8_t* iflag;            /* [B][N]   Aircraft.conflict :278 */
  double* ihs;               /* [B][N][2] intruder (heading, speed), kept only by intruder_turns handles
                                (Simulators/SingleAircraftMCTSRandIntruderEnv.py:322-323); ignored otherwise */
} gca_host_state;

/* Device output buffers of one reset/step.  REAL is double in FAITHFUL mode, float in FAST. */
typedef struct gca_out {
  void* obs;       /* REAL [B][obs_dim]; may be NULL for GCA_OBS_NONE */
  void* achieved;  /* REAL [B][2]  HER kinds only, else NULL */
  void* desired;   /* REAL [B][2]  HER kinds only, else NULL */
  void* reward;    /* REAL [B]     (ignored by gca_reset) */
  uint8_t* done;   /* [B] */
  uint8_t* info;   /* [B] GCA_INFO_* */
  void* nearest;   /* REAL [B] or NULL; shaped_nearest only: dist_nearest_intruder of the step, the value
                      Simulators/SingleAircraftDiscrete3HEREnv.py:178 returns in place of info (9999 if no intruder) */
} gca_out;

/* Recorded draws for GCA_DRAWS_TAPE: env b reads values[b*stride + cursor[b]++]. */
typedef struct gca_tape {
  const double* values; /* device [B][stride] */
  int64_t stride;
  int64_t* cursor;      /* device [B], advanced by the kernels */
} gca_tape;

typedef struct gca_env gca_env;

int gca_abi_version(void);
const char* gca_last_error(void);

/* number of REAL elements of one observation row: 4*N + 8 for VECTOR/RAW, 4*N + 6 for HER/DHER, 6*N + 8 for RAW6,
 * 4 + 5*nearest_n for NEAREST, 0 for NONE */
int gca_obs_dim(const gca_config* cfg, int n_intruders);

/* Replaces B constructions of PKG/SingleAircraftEnv.py:29-43 (and siblings).  Allocates the
 * device state for n_envs environments with n_intruders intruders each on `device`.
 * env_id0 is the global id of env 0 (rank offset for multi-GPU sharding, SURVEY.md 8(e)). */
int gca_create(const gca_config* cfg, int n_envs, int n_intruders, int mode, int draws,
               int device, uint64_t seed, uint32_t env_id0, gca_env** out);
int gca_destroy(gca_env* env);

/* Re-key the Philox stream (gym's seed(); the reference's seed() does not touch its dynamics, Q1). */
int gca_set_seed(gca_env* env, uint64_t seed);

/* Update the parameters in place (the reference re-reads Config inside _get_ob, Q12). */
int gca_set_config(gca_env* env, const gca_config* cfg);

/* reset(): PKG/SingleAircraftEnv.py:66-98 for every env whose mask byte is non-zero
 * (mask == NULL: all).  Writes obs (and achieved/desired); done/info are cleared. */
int gca_reset(gca_env* env, const uint8_t* mask, const gca_tape* tape, const gca_out* out, void* stream);

/* step(action): PKG/SingleAircraftEnv.py:128-184 (+ variants) for all envs in one launch.
 * actions: device int32[B] for the discrete kinds; REAL[B][2] for GCA_ACT_CONTINUOUS2.
 * auto_reset != 0 applies the VecEnv contract (baselines dummy_vec_env.py:52-55): an env that
 * finished is reset in the same launch and `obs` holds the reset observation. */
int gca_step(gca_env* env, const void* actions, const gca_tape* tape, int auto_reset,
             const gca_out* out, void* stream);

/* Number of kernels one gca_step launches for this handle.  GCA_DRAWS_PHILOX: 1 without intruders; else 2 (the main
 * kernel = ownship role + streaming pass, then finish + spawn phase) + 1 for the observation pass of the NEAREST /
 * RAW6 kinds.  GCA_DRAWS_TAPE (parity replays): ownship, streaming pass, finish (+ the observation pass). */
int gca_step_launches(gca_env* env);

/* Synchronises the device and reports a device-side failure of an earlier asynchronous gca_step: GCA_ERR_STATE if a
 * streaming lane gave up waiting for its env's ownship record (the main kernel's ownship role and streaming role
 * hand over through memory inside one launch; the wait is bounded so that a broken assumption fails loudly instead
 * of hanging the GPU).  GCA_OK otherwise.  No reference counterpart. */
int gca_check(gca_env* env);

/* Diagnostics: per-kernel device time of gca_step.  While enabled, every gca_step records CUDA events
 * between its kernels on the caller's stream (do not enable inside a stream capture); gca_profile_read
 * synchronises the device, sums the recorded intervals and clears them.  This is how bench.py times the
 * streaming pass for its roofline line.  The reference has no counterpart (its only timing is the wall
 * clock around a search in Algorithms/MCTS/Agent.py:36-43). */
typedef struct gca_step_profile {
  int64_t steps;
  /* summed over `steps` recorded steps.  GCA_DRAWS_PHILOX (two kernels per step): own_ms = 0, intruders_ms = the
   * main kernel (ownship role + streaming pass), finish_ms = finish + spawn phase, spawn_ms = the nearest-n / turn
   * pass of the variants that have one.  GCA_DRAWS_TAPE: ownship kernel, streaming pass, finish, 0. */
  double own_ms, intruders_ms, finish_ms, spawn_ms;
} gca_step_profile;
int gca_profile_enable(gca_env* env, int on);
int gca_profile_read(gca_env* env, gca_step_profile* out);

/* Same step driven from HOST memory (the end-to-end path): copies actions host->device,
 * launches, copies obs/reward/done/info device->host into `host_out` (host pointers with the
 * same shapes; pinned memory recommended) and synchronises.  PHILOX draws only. */
int gca_step_host(gca_env* env, const void* actions_host, int auto_reset, const gca_out* host_out);
int gca_reset_host(gca_env* env, const gca_out* host_out);
/* The asynchronous form (VecEnv.step_async / step_wait of baselines common/vec_env/__init__.py:76-100): _begin enqueues
 * the upload of the actions, the step and the download of its outputs into `host_out` and returns; _wait blocks until
 * the outputs of the OLDEST step begun and not yet waited for are in host memory.  Two steps may be in flight: the
 * device-side outputs are double-buffered and the download runs on a stream of its own, so the download of step t
 * overlaps the kernels of step t + 1 (give the two steps different host buffers; `actions_host` must stay valid until
 * the matching _wait).  gca_step_host = _begin + _wait.  A handle driven through the host path must not also be
 * driven through gca_step / gca_reset on another stream without a device synchronisation in between: the host path
 * orders its work on its own streams. */
int gca_step_host_begin(gca_env* env, const void* actions_host, int auto_reset, const gca_out* host_out);
int gca_step_host_wait(gca_env* env);

/* _get_ob() of the current state without stepping (PKG/SingleAircraftEnv.py:100-126). */
int gca_observe(gca_env* env, const gca_out* out, void* stream);

/* Per-env counters without a host round trip: device int32 [n_envs][4] = (no_conflict - the attribute
 * Algorithms/MCTS/Agent.py:52 reads after an episode -, steps of the current episode, Philox tick, finished
 * episodes).  Asynchronous device-to-device copy on `stream`. */
int gca_read_counters(gca_env* env, int32_t* counters, void* stream);

/* Full-state access (teacher-forced parity, MCTS root states, checkpointing).  Synchronous.
 * NULL members of the view are skipped. */
int gca_get_state(gca_env* env, const gca_host_state* dst);
int gca_set_state(gca_env* env, const gca_host_state* src);

/* HER relabelling reward, PKG/SingleAircraftHEREnv.py:194-196 (kind GCA_OBS_HER:
 * -(d > radius), always -0.0f for normalised goals, Q14) and
 * PKG/SingleAircraftDiscreteHEREnv.py:184-186 (kind GCA_OBS_DHER: d < radius).
 * ag, g: device [m][2], f64 when is_f64 else f32; out: device float[m]. */
int gca_compute_reward(const void* ag, const void* g, int64_t m, double radius, int kind,
                       int is_f64, float* out, int device, void* stream);
/* The same with the achieved goals repeating: ag [n_ag][2], g [m][2], m = k * n_ag, out[i] = reward(ag[i % n_ag], g[i]) -
 * the relabel of DDPG.py:308-315 (k substitute goals per transition) without materialising the k copies of ag. */
int gca_compute_reward_tiled(const void* ag, int64_t n_ag, const void* g, int64_t m, double radius, int kind, int is_f64,
                             float* out, int device, void* stream);

/* compute_input_reward(new_inputs) of Simulators/SingleAircraftDiscrete9HEREnv.py:244-276, the reward the repo's own
 * HER learner gives a relabelled transition (Algorithms/pytorch/agent_her.py:107-117), for m rows at once.
 * rows: device [m][dim] (observation + desired goal: own x, y at 0-1, the listed intruders from entry 4 on, read with
 * the reference's stride of 4, the goal in the last two entries), f64 when is_f64 else f32.  out: device double[m]
 * (the reference returns Python floats); done (nullable): device uint8[m], r == 10 or r == -10 (agent_her.py:117). */
typedef struct gca_input_reward_cfg {
  double window_width, window_height;     /* Config.window_width / window_height (the un-normalisation) */
  double minimum_separation, nmac_dist, goal_radius;
  double conflict_penalty, nmac_penalty, goal_reward, step_penalty;
  int32_t n_listed;                       /* Config.n */
  int32_t has_intruders;                  /* Config.intruder_size != 0 */
  int32_t sparse_reward;                  /* Config.sparse_reward */
  int32_t reserved;
} gca_input_reward_cfg;
int gca_input_reward(const void* rows, int64_t m, int dim, int is_f64, const gca_input_reward_cfg* cfg, double* out,
                     uint8_t* done, int device, void* stream);

/* ------------------------------------------------------------------------------------------
 * MCTS forward model (Algorithms/MCTS/nodes_single.py) - batched device-side playouts.
 * Parameters follow Algorithms/MCTS/config_single.py:4-64. */
typedef struct gca_mcts_config {
  double window_width, window_height;
  double minimum_separation;          /* conflict AND goal radius of the model (nodes_single.py:87,95; Q24) */
  double min_speed, max_speed, d_speed, speed_sigma, position_sigma;
  double d_heading, heading_sigma;
  int32_t simulate_frame;             /* sub-frames per move() (config_single.py:59) */
  int32_t search_depth;               /* moves per playout (config_single.py:61) */
  /* Algorithms/MCTS/nodes_single_randintru.py (the model of Agent_RandInt.py): state vectors are the 6 N + 8 raw
   * observation of Simulators/SingleAircraftMCTSRandIntruderEnv.py (x, y, vx, vy, speed, heading per intruder); ALL N
   * intruders are seen ((len - 8) // 6, :47); after its advance every intruder draws np.random.random() and, below
   * turn_prob, turns by radians(uniform(-turn_max_deg, turn_max_deg)) - f64 velocity = speed * (cos, sin) (:64-71);
   * the speed clamp reads the speed itself (:74, the index bug Q23 of nodes_single.py is fixed there). */
  int32_t random_intruders;
  int32_t reserved0;
  double turn_prob;                   /* 0.1 (:64) */
  double turn_max_deg;                /* 10 (:65) */
} gca_mcts_config;

/* Philox counter of the playout kernels: (root id, playout id, what, index) */
#define GCA_MCTS_DRAW_ACTION 0u       /* index = move number: action = floor(9 * u) */
#define GCA_MCTS_DRAW_HEADING 1u      /* index = global sub-frame: Box-Muller cos branch * heading_sigma */
#define GCA_MCTS_DRAW_SPEED 2u        /* index = global sub-frame (only drawn when speed_sigma != 0) */
#define GCA_MCTS_DRAW_INTRUDER 3u     /* + intruder index; index = global sub-frame (only when position_sigma != 0) */
#define GCA_MCTS_DRAW_TURN 0x40000000u /* + intruder index; index = global sub-frame: (p, u) of a random_intruders turn */

enum { GCA_MCTS_WALL = 1, GCA_MCTS_CONFLICT = 2, GCA_MCTS_GOAL = 4 };

/* ---- episode statistics (baselines common/vec_env/vec_monitor.py:21-37 VecMonitor.step_wait, bench/monitor.py:54-78):
 * ep_return += reward (float32 accumulation, like np.zeros(num_envs, 'f')), ep_length += 1, and for every finished env
 * a record (env, length, return, step) is appended to a ring on the device and its accumulators restart at 0 - no
 * host synchronisation per step; the host drains the ring whenever it likes.  reward: REAL [n_envs] as written by
 * gca_step (is_f64 = FAITHFUL mode); ring_count: device counter of all records ever appended (slot = count % cap). */
typedef struct gca_episode_record {
  int32_t env;
  int32_t length;
  float ep_return;
  uint32_t step;
} gca_episode_record;

int gca_monitor_update(const void* reward, int is_f64, const uint8_t* done, int64_t n_envs, float* ep_return,
                       int32_t* ep_length, gca_episode_record* ring, int64_t ring_capacity,
                       unsigned long long* ring_count, uint32_t step, int device, void* stream);

/* Batch-wide counters for the optional statistics reduce across GPUs (SURVEY 8(e); the figures Algorithms/MCTS/Agent.py:55-62
 * prints): stats[GCA_STAT_*] += ... over the n_envs envs of one step.  info: the GCA_INFO_* codes gca_step wrote.
 * stats: device uint64 [GCA_STAT_COUNT], accumulated with one atomic per warp and counter. */
enum { GCA_STAT_STEPS = 0, GCA_STAT_EPISODES = 1, GCA_STAT_NMAC = 2, GCA_STAT_CONFLICT_STEPS = 3, GCA_STAT_GOAL = 4,
       GCA_STAT_WALL = 5, GCA_STAT_MAXSTEPS = 6, GCA_STAT_COUNT = 8 };
int gca_stats_update(const uint8_t* done, const uint8_t* info, int64_t n_envs, unsigned long long* stats, int device,
                     void* stream);

/* ---- HER replay: the "future" relabelling sampler of baselines (Algorithms/baselines-master/baselines/her/
 * her_sampler.py:19-61 _sample_her_transitions, called by replay_buffer.py:sample with o_2 = o[:, 1:], ag_2 = ag[:, 1:])
 * on an episode buffer that lives on the device.  For each of `batch` transitions: episode e and time t are drawn,
 * rows o[e][t], u[e][t], g[e][t], ag[e][t], o_2 = o[e][t+1], ag_2 = ag[e][t+1] are gathered, with probability
 * future_p = 1 - 1 / (1 + replay_k) the goal is replaced by ag[e][t + 1 + int(u * (T - t))], and the reward is
 * recomputed by the env's compute_reward(ag_2, g) (reward_kind GCA_OBS_HER / GCA_OBS_DHER, goals are 2-D).
 * All arrays are REAL = double (is_f64, what baselines' numpy buffers hold) or float. */
typedef struct gca_her_episodes {
  const void* o;  /* REAL [n_episodes][T+1][dim_o] */
  const void* u;  /* REAL [n_episodes][T][dim_u] */
  const void* g;  /* REAL [n_episodes][T][dim_g] */
  const void* ag; /* REAL [n_episodes][T+1][dim_g] */
} gca_her_episodes;

/* the four np.random calls of the sampler, in call order, as device arrays of length batch; a NULL gca_her_draws*
 * means Philox: counter (b & 0xffffffff, b >> 32, call, block), block 0 -> (episode, t) = (int(u0 * E), int(u1 * T)),
 * block 1 -> (u_her, u_offset) */
typedef struct gca_her_draws {
  const int64_t* episode_idxs; /* np.random.randint(0, rollout_batch_size, batch_size) */
  const int64_t* t_samples;    /* np.random.randint(T, size=batch_size) */
  const double* u_her;         /* np.random.uniform(size=batch_size) < future_p */
  const double* u_offset;      /* np.random.uniform(size=batch_size) * (T - t_samples) */
} gca_her_draws;

typedef struct gca_her_transitions {
  void *o, *u, *g, *ag, *o_2, *ag_2; /* REAL [batch][dim] */
  float* r;                          /* [batch] */
  int32_t *episode, *t, *future_t;   /* [batch] (nullable) what was drawn; future_t = -1 where the goal was kept */
} gca_her_transitions;

int gca_her_sample(const gca_her_episodes* episodes, int64_t n_episodes, int T, int dim_o, int dim_u, int dim_g,
                   int is_f64, int64_t batch, double future_p, double goal_radius, int reward_kind,
                   const gca_her_draws* draws, uint64_t seed, uint32_t call, const gca_her_transitions* out, int device,
                   void* stream);

/* SingleAircraftState.move(action) for m independent states (nodes_single.py:39-100; with cfg->random_intruders
 * nodes_single_randintru.py:39-116 on [m][6N+8] vectors, tape order per intruder: normal, normal, random(), [uniform]).
 * states: device double [m][4N+8] raw observation vectors (Simulators/SingleAircraftMCTSEnv.py:98-124),
 * advanced in place; actions: device int32 [m] (a0*3+a1); flags: device uint8 [m] (GCA_MCTS_* bits).
 * tape (nullable): the model's np.random.normal values in call order, values[i*stride + cursor[i]++];
 * without a tape the draws are Philox (seed; root id = id0 + i, playout id 0). */
int gca_mcts_move(const gca_mcts_config* cfg, int n_intruders, double* states, const int32_t* actions,
                  uint8_t* flags, int64_t m, const gca_tape* tape, uint64_t seed, uint32_t id0, int first_frame,
                  int device, void* stream);

/* Node.rollout(search_depth) from n_roots root states, `playouts` independent random playouts each
 * (nodes_single.py:198-204, common.py:54-55): uniform actions until terminal or `depth` moves, reward()
 * of the final state (nodes_single.py:25-32).  first_action (nullable, int8 [n_roots][playouts], -1 =
 * random) forces the first move, which is how a tree policy hands its selected child to the playout.
 * Outputs: rewards double [n_roots][playouts]; first_out int8 (the first action taken);
 * flags uint8 (GCA_MCTS_* of the final state). */
int gca_mcts_playouts(const gca_mcts_config* cfg, int n_intruders, const double* roots, int64_t n_roots,
                      int playouts, int depth, const int8_t* first_action, uint64_t seed, uint32_t root_id0,
                      double* rewards, int8_t* first_out, uint8_t* flags, int device, void* stream);

/* MCTS(root).best_action(simulations, search_depth) for n_roots independent roots, the whole UCT tree resident on
 * the device (search_single.py:8-22 best_action / tree_policy; common.py:47-52 best_child with c = 1.4 in the
 * tree and c = 0 for the final pick; nodes_single.py:188-193 expand - untried actions popped from the end -,
 * :198-204 rollout, :206-210 backpropagate; Algorithms/MCTS/Agent.py:37-41 is the call site this replaces).
 * Requires cfg->position_sigma == 0 (config_single.py:27) and no random_intruders: the model's intruders then move on
 * root-only trajectories and a tree node is just the ownship (GCA_ERR_STATE otherwise: the drop-in node classes then
 * run the tree on the host with device move / rollout).  Draws are Philox, keyed (seed; root id = root_id0 + r,
 * simulation index, GCA_MCTS_DRAW_*, global sub-frame).
 * workspace: device scratch of gca_mcts_search_workspace(...) bytes, caller-owned, 16-byte aligned.
 * Outputs (device): best_action int32 [n_roots] (a0*3+a1 of the most valuable root child, -1 if simulations == 0);
 * child_n, child_q double [n_roots][9] and child_action int32 [n_roots][9] (nullable): visit count, value sum and
 * action of the root's children in creation order (unused slots 0 / 0 / -1). */
int64_t gca_mcts_search_workspace(const gca_mcts_config* cfg, int n_intruders, int64_t n_roots, int simulations,
                                  int depth);
int gca_mcts_search(const gca_mcts_config* cfg, int n_intruders, const double* roots, int64_t n_roots,
                    int simulations, int depth, uint64_t seed, uint32_t root_id0, void* workspace,
                    int64_t workspace_bytes, int32_t* best_action, double* child_n, double* child_q,
                    int32_t* child_action, int device, void* stream);

/* ------------------------------------------------------------------------------------------
 * Image observation of SingleAircraftStackEnv (PKG/SingleAircraftStackEnv.py:104-114, 179-214):
 * render() -> 800x800 RGB frame (white clear; ownship, goal, intruders drawn in that order as 32x32
 * textured quads rotated by heading - pi/2, src-alpha blending into an 8-bit framebuffer), then
 * cv2.cvtColor(RGB2GRAY) and cv2.resize(INTER_AREA) by 4 -> uint8 [H/4][W/4], row 0 = top.
 * The full-resolution frame is never materialised: each output pixel evaluates its 16 samples
 * against the few sprites whose bounding box touches its cell.  DESIGN.md section 4.5 is the spec
 * (the GL half of the reference cannot run without a display, so the restatement is the spec).
 *
 * sprites: device uint8 [3][32][32][4] = (ownship, goal, intruder) x rows top->bottom x RGBA, 4-byte aligned.
 * frames : device uint8, 4-byte aligned; env b writes (H/4)*(W/4) bytes at frames + b*env_stride + slot*plane_stride.
 *          env_stride and plane_stride are multiples of 4.  When frames, both strides and the plane size are
 *          multiples of 16 a plane leaves with one bulk copy, otherwise with 4-byte stores (same bytes).
 * clear_mask (nullable, device uint8 [B]): for a non-zero entry the other n_planes-1 planes of that env
 * are zero-filled first - VecFrameStack's reset of a finished env (vec_frame_stack.py:19-23, Q21).
 * GCA_ERR_INVALID for an unaligned pointer or stride; GCA_ERR_STATE for a window whose width is not a multiple
 * of 16 or height not a multiple of 4, and for one whose output plane, with about 70 KB of textures and tables,
 * does not fit in the 227 KB of shared memory a block may use (1600x1504 fits, 1600x1600 does not).  Neither
 * launches a kernel. */
#define GCA_RASTER_MAX_INTRUDERS 126
int gca_raster(gca_env* env, const uint8_t* sprites, uint8_t* frames, int64_t env_stride, int64_t plane_stride,
               int n_planes, int slot, const uint8_t* clear_mask, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GCA_H_ */

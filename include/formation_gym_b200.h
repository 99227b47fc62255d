/*
 * formation_gym_b200.h -- C ABI of the B200-native MPE step path for jc-bao/gym-formation.
 *
 * The reference has no native layer: its hot path is per-object Python (formation_gym/
 * environment.py:113-142 -> formation_gym/core.py:206-322 -> formation_gym/envs/
 * formation_hd_env.py:38-75 / basic_formation_env.py:29-52).  This header declares the entry
 * points a maintainer of the reference would bind (ctypes stub in INTEGRATION.md) to replace
 * those functions with sm_100a kernels.  Each entry cites the reference code it replaces.
 *
 * Conventions
 *  - Every buffer is CALLER-OWNED DEVICE memory (plain pointers; no torch types).  The library
 *    allocates nothing persistent, keeps no global state and never frees caller memory.
 *  - All work is enqueued asynchronously on `stream` (a cudaStream_t passed as void*; NULL is
 *    the legacy default stream).  No internal synchronisation, no hidden streams.  Entry points
 *    are re-entrant and may be called from several host threads on different streams/buffers.
 *  - Layout is the reference's VecEnv contract (train/maddpg-v2/utils/env_wrappers.py:68-72),
 *    env-major, contiguous:  pos/vel [E,N,2]  act [E,N,act_dim]  comm [E,N,2]  obs [E,N,D]
 *    reward [E,N,1]  indiv [E,N]  done [E,N] (uint8)  step [E] (int32)  ideal_shape [E,N,2]
 *    ideal_vel [E,2]  landmarks [E,L,2].   hd: L = N, D = 6N.  basic: D = 4 + 2L + 4(N-1).
 *    hd_partial: D = 2 + 2L + 2 num_obs + 2(N-1).  hd_partial_range: D = 2 + 2L + 4(N-1).
 *    hd_obstacle: D = 2 + 2L + 4(N-1) (L = goal landmarks + obstacles).
 *    act_dim = 2 for silent agents (both target scenarios), 2 + 2 when params.silent == 0.
 *  - `float` entry points compute in fp32, the `_f64` twins in fp64 with FMA contraction
 *    disabled (the 25-step 1e-9 parity build).  Same semantics otherwise.
 *  - Return value: 0 on success; < 0 on error (FG_ERR_*), message via fg_last_error()
 *    (thread-local).  No C++ exception crosses the ABI.  NaNs propagate exactly as in the
 *    reference (coincident agents -> 0/0, core.py:312); no epsilon is added anywhere.
 *  - The caller's `act` buffer is never written (the reference's in-place `u *= sensitivity`
 *    on the caller's array, environment.py:216-221, is deliberately not reproduced).
 *  - RNG: counter-based Philox4x32-10, key = seed, counter = (global env id, agent, tick,
 *    purpose); tick = the `tick` argument + fg_buffers.tick_dev[0] when that pointer is given.  `env_offset` is the global index of env 0 of this buffer, so results do not
 *    depend on launch geometry or on how envs are sharded over GPUs.  The caller supplies a
 *    fresh `tick` per call (e.g. a global step counter).  Parity with the reference's global
 *    MT19937 stream (np.random.*) is statistical only.
 */
#ifndef FORMATION_GYM_B200_H
#define FORMATION_GYM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FG_ABI_VERSION 9
#define FG_MAX_AGENTS 256      /* one CTA holds at least one whole env; 3^5 = 243 fits */
#define FG_MAX_LANDMARKS 256
#define FG_MAX_WALLS 8

#define FG_OK 0
#define FG_ERR_ARG (-1)        /* null pointer, bad size, unsupported combination */
#define FG_ERR_CUDA (-2)       /* launch / runtime failure, see fg_last_error() */

/* scenario ids */
#define FG_SCENARIO_HD 0       /* formation_gym/envs/formation_hd_env.py */
#define FG_SCENARIO_BASIC 1    /* formation_gym/envs/basic_formation_env.py */
#define FG_SCENARIO_HD_PARTIAL 2        /* formation_gym/envs/formation_hd_partial_env.py: obs = [p_vel, landmark
                                           positions (absolute), p_j - p_i of the next num_obs agents (cyclic), comm];
                                           reward = -Hausdorff(agents - mean, landmarks - mean) - #collisions (s1+s2) */
#define FG_SCENARIO_HD_PARTIAL_RANGE 3  /* formation_gym/envs/formation_hd_partial_range_env.py: as above with
                                           other_pos of ALL others clipped to [-obs_range, obs_range] */

#define FG_SCENARIO_HD_OBSTACLE 4       /* formation_gym/envs/formation_hd_obs_env.py: the last num_obstacles entries of
                                           `landmarks` are movable COLLIDING obstacles (agent-obstacle and
                                           obstacle-obstacle contact forces, integrated like agents, core.py:240-277);
                                           obs = [p_vel, goal landmarks (absolute), obstacles - p_i, p_j - p_i, comm];
                                           reward = -Hausdorff(agents - mean, goals - mean) - 2 per agent collision
                                           (s1+s2) - 2 per obstacle collision; the reward hook's side effect sets every
                                           obstacle's velocity to (0, obstacle_fall_vy) above obstacle_floor, else 0 */

/* core.Wall (formation_gym/core.py:27-41) */
typedef struct fg_wall {
    int32_t orient;            /* 0 = 'H' (lies along x at y = axis_pos), 1 = 'V' */
    int32_t hard;
    double axis_pos, end0, end1, width;
} fg_wall;

/* World / Agent constants (formation_gym/core.py:45-110,112-139; environment.py:218-221). */
typedef struct fg_params {
    double dt;                 /* core.py:125  0.1 */
    double damping;            /* core.py:127  0.25 */
    double contact_force;      /* core.py:129  1e2 */
    double contact_margin;     /* core.py:130  1e-3 */
    double sensitivity;        /* environment.py:218  5.0 (replaced by accel when has_accel) */
    double agent_size;         /* hd 0.03 (formation_hd_env.py:26), basic 0.1 */
    double mass;               /* core.py:69  1.0 */
    double accel;              /* core.py:65  used iff has_accel (scales the action twice) */
    double max_speed;          /* core.py:64  used iff has_max_speed */
    double u_noise;            /* core.py:97  0 = off (None) */
    double c_noise;            /* core.py:99  0 = off (None) */
    double obs_range;          /* FG_SCENARIO_HD_PARTIAL_RANGE: Scenario.obs_range (formation_hd_partial_range_env.py:15) */
    double obstacle_size;      /* FG_SCENARIO_HD_OBSTACLE: 0.15 (formation_hd_obs_env.py:44) */
    double obstacle_mass;      /* Entity.initial_mass 1.0 (core.py:69) */
    double obstacle_floor;     /* -2.2 (formation_hd_obs_env.py:86) */
    double obstacle_fall_vy;   /* -1.0 (formation_hd_obs_env.py:87) */
    int32_t has_accel;
    int32_t has_max_speed;
    int32_t collide;           /* agents collide (formation_hd_env.py:24) */
    int32_t silent;            /* 1: comm state = 0 (core.py:281-282); 0: c = action.c + noise */
    int32_t world_length;      /* episode length; done = step >= world_length */
    int32_t n_walls;
    int32_t action_prescaled;  /* 1: `act` already is agent.action.u (after _set_action), i.e. World.step()
                                  called on its own (core.py:206); the sensitivity multiply is skipped */
    int32_t num_obs;           /* FG_SCENARIO_HD_PARTIAL: Scenario.num_obs (formation_hd_partial_env.py:15) */
    int32_t num_obstacles;     /* FG_SCENARIO_HD_OBSTACLE: Scenario.num_obstacles (formation_hd_obs_env.py:14); the
                                  entry points' L counts goal landmarks + obstacles */
    int32_t num_landmarks;     /* fg_world_step only (it has no L argument): entries per env of `landmarks` /
                                  `landmark_vel` when num_obstacles > 0 -- World.step on a world whose trailing
                                  num_obstacles landmarks are movable colliders (core.py:240-277) */
    /* optional per-agent DEVICE arrays [N] in the entry point's real type; NULL = scalar above.
       agent_accel / agent_max_speed entries < 0 mean "None" for that agent. */
    const void* agent_mass;
    const void* agent_size_arr;
    const void* agent_accel;
    const void* agent_max_speed;
    fg_wall walls[FG_MAX_WALLS];
} fg_params;

/* Device buffers of one env batch (all caller-owned; element type = entry point's real type
   unless stated).  Pointers marked (opt) may be NULL. */
typedef struct fg_buffers {
    void* pos;                 /* [E,N,2]  in/out  agent.state.p_pos */
    void* vel;                 /* [E,N,2]  in/out  agent.state.p_vel */
    const void* act;           /* [E,N,act_dim] in; unused when random actions are requested */
    void* comm;                /* (opt) [E,N,2] out  agent.state.c */
    void* ideal_shape;         /* hd: [E,N,2] Scenario.ideal_shape (centred; formation_hd_env.py:93) */
    void* ideal_vel;           /* hd: [E,2]   Scenario.ideal_vel   (formation_hd_env.py:95) */
    void* landmarks;           /* basic: [E,L,2] required.  hd: (opt) [E,N,2] in/out, re-centred on the
                                  agents' centroid as the reference's observation side effect does
                                  (formation_hd_env.py:40-44; visualisation only) */
    int32_t* step;             /* [E] in/out  env.current_step */
    void* obs;                 /* (opt) [E,N,D] out; NULL = state+reward only */
    void* reward;              /* [E,N,1] out  shared reward sum_i r_i (environment.py:136-138) */
    void* indiv;               /* (opt) [E,N] out  info['individual_reward'] (environment.py:130) */
    uint8_t* done;             /* [E,N] out  (environment.py:172-177) */
    void* ep_return;           /* (opt) [E] in/out running episode return (shared reward) */
    int32_t* ep_collisions;    /* (opt) [E] in/out running count of reward-collisions */
    double* stats;             /* (opt) [4] in/out: n_episodes, sum return, sum return^2,
                                  sum collisions -- updated atomically at episode ends */
    void* landmark_vel;        /* FG_SCENARIO_HD_OBSTACLE: (opt) [E,L,2] in/out landmark.state.p_vel; only the obstacle
                                  entries are read and written (NULL: obstacles start the step at rest) */
    uint32_t* tick_dev;        /* (opt) [2] in/out, zero-initialised by the caller: [0] is ADDED to the
                                  `tick` argument of every entry point; fg_world_step / fg_step_fused
                                  advance it by the number of env steps they ran ([1] is their arrival
                                  counter).  Lets a CUDA graph of step launches be replayed with fresh
                                  random numbers although its kernel arguments are frozen. */
    const void* contact_pos;   /* (opt) [E,N,2] in: World.cache_dists (core.py:132,224-225,298-301).  With the cache on, the
                                  reference's contact forces use the distances stored at the END of the previous
                                  World.step -- i.e. the positions of that moment, which differ from the current ones
                                  only if the state was edited in between (or after a reset without a fresh
                                  calculate_distances()).  Those positions go here; NULL = current positions.
                                  fg_world_step / fg_step_fused, agents only (no movable obstacles). */
    uint8_t* nan_flag;         /* (opt) [E] in/out, zero-initialised by the caller: set to 1 (and never cleared by
                                  the library) when, after a step's physics, the env holds a non-finite position --
                                  the reference's documented failure mode (coincident agents -> 0/0 in core.py:312,
                                  NaN state and rewards until the next reset; train/README.md:194-197).  Written by
                                  fg_step_fused and fg_obs_reward; costs no traffic while every env is finite. */
} fg_buffers;

/* Target bank of formation_hd_env (the *_targets entry points): `count` = K formation tasks, DEVICE arrays in the entry
 * point's real type.  At every reset of env e -- fg_reset_targets and the in-kernel auto-reset alike -- the env takes
 * task k = index[e] when index is given and 0 <= index[e] < K, else k drawn uniformly from Philox (purpose 6,
 * umulhi(x, K)).  shapes[k] replaces the uniform landmark draw of reset_world (formation_hd_env.py:89) and is centred
 * with the same arithmetic (ideal_shape = raw - mean(raw), :93; tracked landmarks receive the raw entry); vels[k], when
 * given, replaces the ideal_vel draw (:95).  Positions, velocities, comm, step and the episode accumulators take the
 * same draws as without a bank.  Scenario.generate_shape (formation_hd_env.py:123-139) gives hierarchical entries. */
typedef struct fg_targets {
    const void* shapes;        /* [K,N,2] raw target shapes */
    const void* vels;          /* (opt) [K,2] target ideal velocities; NULL = drawn as without a bank */
    const int32_t* index;      /* (opt) [E] task per env, read at each reset (a curriculum may rewrite it between
                                  calls, in stream order); an entry outside [0, K) -- e.g. -1 -- means "draw" */
    int32_t count;             /* K >= 1 */
} fg_targets;

/* Terminal block (the *_final entry points): caller-owned DEVICE arrays in the entry point's real type, shaped like the
 * state arrays.  When a single-step call with auto_reset ends env e's episode, the kernel copies env e's post-step
 * state -- what the call returns with auto_reset == 0 -- into the block before the auto-reset overwrites it.  Entries
 * of envs whose episode did not end are not written; the mask of written envs is the step's own done[e*N].  Every
 * episode ends on the time limit (environment.py:172-177), so this is the state s_T a trainer bootstraps V(s_T) from
 * (baselines' infos[e]['terminal_observation']; fg_final_obs below). */
typedef struct fg_final {
    void* pos;                 /* [E,N,2] */
    void* vel;                 /* [E,N,2] */
    void* comm;                /* [E,N,2], non-silent agents only (ignored for silent ones) */
    void* ideal_shape;         /* [E,N,2], formation_hd_env only */
    void* ideal_vel;           /* [E,2], formation_hd_env only */
    void* landmarks;           /* [E,L,2], every other scenario (formation_hd_obs_env: goals, then the obstacles at their
                                  post-step positions) */
} fg_final;

int fg_abi_version(void);
const char* fg_last_error(void);

/* A/B switches for tests and profiling (never needed in production; defaults select the product kernels).  They are
 * process-global, read once from the environment variables FG_<NAME IN UPPER CASE> when the library is first used
 * (never on the launch path) and can be changed at run time here.  Names and ranges:
 *   force_tile_kernel 0/1  fg_step_fused always takes the generic tile kernels instead of the warp-autonomous ones
 *                          (formation_hd_env / basic: k_hd_warp; partial, partial_range, obs_env: k_lm_warp)
 *   no_fast_pairs 0/1      tile kernel: scalar pair loops instead of the packed ones (N >= 32)
 *   force_fast_pairs 0/1   tile kernel: packed pair loops also for 32 <= N < 64 with observations
 *   no_cells 0/1           packed pair loops: O(N^2) group filters instead of the hashed cell lists
 *   row_chunks 0/1/2       long-row observation writer: per-row pieces with the static 2/3 from a shared image /
 *                          whole rows staged 4-128 at a time with one bulk store per chunk for N <= 80 (default) /
 *                          chunks for every N
 *   row_min_n 3..256       bulk-store row writers (formation_hd_env, silent agents) from this agent count up (10)
 *   row_chunk_max_log2 1..7  chunked writer: at most 2^k rows per chunk (7; the image is also capped at 32 KB)
 *   row_nbuf 1/2           per-row pieces: staging buffers per warp
 *   no_early_rows 0/1      long-row observation writer: rows leave after the reward pass
 *   no_tile_image 0/1      short-row observation writer: flat item loop instead of the tile image
 *   no_std_kernel 0/1      warp kernels: never the instantiation specialised for the standard configuration (fp32
 *                          k_lm_warp has no other: the partial / obstacle scenarios then take the tile kernels)
 *   l2_prefetch 0/1/2      warp kernel: prefetch.global.L2 of the state two spans ahead: never / when the state
 *                          arrays exceed ~1/3 of L2 (default) / always
 *   pf_spans 2..8          ... how many spans ahead (2)
 *   waves 1..64            warp kernel: grid = waves x one resident wave
 *   nvtx 0/1               NVTX ranges (domain-less, named after the entry point) around every launch
 * Unknown names / out-of-range values return FG_ERR_ARG. */
int fg_set_option(const char* name, int value);
int fg_get_option(const char* name, int* value);
/* SM count and compute capability of the current device (host logic sizes grids with it). */
int fg_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* World.step (formation_gym/core.py:206-225) preceded by MultiAgentEnv._set_action
 * (environment.py:187-236): apply_action_force (core.py:228-237, Philox u-noise),
 * apply_environment_force / get_entity_collision_force (core.py:240-262,289-322; walls
 * 325-362), integrate_state (core.py:264-277), update_agent_state (core.py:279-286).
 * Reads b->pos, vel, act; writes pos, vel, comm.  One fused kernel.
 * With p->num_obstacles > 0 the trailing obstacles of b->landmarks [E, p->num_landmarks, 2] take part in the contact
 * forces and are integrated too (their velocities in b->landmark_vel, in/out). */
int fg_world_step(const fg_params* p, const fg_buffers* b, int E, int N,
                  uint64_t seed, uint32_t tick, uint32_t env_offset, void* stream);
int fg_world_step_f64(const fg_params* p, const fg_buffers* b, int E, int N,
                      uint64_t seed, uint32_t tick, uint32_t env_offset, void* stream);

/* Scenario.observation + Scenario.reward from the CURRENT state, for every agent of every env
 * (formation_hd_env.py:38-75,119-121 / basic_formation_env.py:29-52,89-91) plus the shared
 * reward sum (environment.py:136-138).  Writes obs, reward, indiv (and hd landmarks).
 * Does not touch step/done. */
int fg_obs_reward(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L,
                  void* stream);
int fg_obs_reward_f64(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L,
                      void* stream);

/* MultiAgentEnv.step (environment.py:113-142) fused into ONE launch: _set_action, World.step,
 * observation, reward, done, shared-reward sum, episode statistics and (auto_reset != 0) the
 * VecEnv auto-reset (train/maddpg-v2/utils/env_wrappers.py:14-18: when the episode ends the
 * terminal reward/done are returned together with the RESET observation).
 * n_steps > 1 runs a whole rollout inside the kernel with state held on chip; then actions are
 * drawn in-kernel from the random policy U(-1,1) (test.py:20) and b->act is ignored.
 * n_steps == 1 and random_actions == 0 is the plain step on caller-provided actions.
 * random_actions == 2: as 1, and the drawn actions are also WRITTEN to b->act [E,N,2] (with fg_step_policy the one case
 * in which the library writes that buffer) so that the caller has the (obs, action, reward) triple of the step -- the random
 * policy and the step in one launch instead of fg_random_actions + fg_step_fused. */
int fg_step_fused(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L,
                  int n_steps, int random_actions, int auto_reset,
                  uint64_t seed, uint32_t tick, uint32_t env_offset, void* stream);
int fg_step_fused_f64(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L,
                      int n_steps, int random_actions, int auto_reset,
                      uint64_t seed, uint32_t tick, uint32_t env_offset, void* stream);

/* Scenario.reset_world (formation_hd_env.py:77-95 / basic_formation_env.py:54-65) +
 * MultiAgentEnv.reset's current_step = 0 (environment.py:145) for envs with mask[e] != 0
 * (mask NULL = all).  Draw order per env follows the reference: agents, landmarks, ideal_vel.
 * Writes pos, vel(=0), comm(=0), landmarks, ideal_shape, ideal_vel, step(=0), ep_return(=0). */
int fg_reset(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L,
             const uint8_t* mask, uint64_t seed, uint32_t tick, uint32_t env_offset, void* stream);
int fg_reset_f64(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L,
                 const uint8_t* mask, uint64_t seed, uint32_t tick, uint32_t env_offset,
                 void* stream);

/* fg_reset / fg_step_fused / fg_step_policy with a target bank (fg_targets above): every reset the call performs --
 * the masked reset, or the auto-reset of an env whose episode ends -- takes the env's task from the bank.  Everything
 * else is the plain entry point's; t == NULL is exactly the plain entry point (which is this call with NULL).
 * FG_ERR_ARG unless scenario == FG_SCENARIO_HD, t->count >= 1, t->shapes != NULL and shapes / vels are 8-byte (fp32)
 * / 16-byte (fp64) aligned (index: 4-byte). */
int fg_reset_targets(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L,
                     const uint8_t* mask, uint64_t seed, uint32_t tick, uint32_t env_offset, void* stream,
                     const fg_targets* t);
int fg_reset_targets_f64(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L,
                         const uint8_t* mask, uint64_t seed, uint32_t tick, uint32_t env_offset, void* stream,
                         const fg_targets* t);
int fg_step_fused_targets(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L,
                          int n_steps, int random_actions, int auto_reset,
                          uint64_t seed, uint32_t tick, uint32_t env_offset, void* stream, const fg_targets* t);
int fg_step_fused_targets_f64(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L,
                              int n_steps, int random_actions, int auto_reset,
                              uint64_t seed, uint32_t tick, uint32_t env_offset, void* stream, const fg_targets* t);

/* World.calculate_distances (formation_gym/core.py:156-180), the distance cache behind World.cache_dists, for every env:
 * ent_pos [E,M,2] entity positions in world.entities order (agents, then landmarks), ent_size [M] ->
 * dist_vect [E,M,M,2] (p_a - p_b above the diagonal, the negative below), dist_mag [E,M,M]
 * (np.linalg.norm(..., axis=2)), collisions [E,M,M] uint8 (dist_mag <= min_dists; True on the diagonal, as in the
 * reference), min_dists [M,M] (size_a + size_b, 0 on the diagonal). */
int fg_pair_distances(const void* ent_pos, const void* ent_size, int E, int M, void* dist_vect, void* dist_mag,
                      uint8_t* collisions, void* min_dists, void* stream);
int fg_pair_distances_f64(const void* ent_pos, const void* ent_size, int E, int M, void* dist_vect, void* dist_mag,
                          uint8_t* collisions, void* min_dists, void* stream);

/* Random policy: act[e,i,:] ~ U(-1,1) (test.py:20 -> Box.sample, environment.py:67-68), same
 * Philox stream the in-kernel rollout uses, so step-by-step and in-kernel rollouts agree. */
int fg_random_actions(void* act, int E, int N, uint64_t seed, uint32_t tick, uint32_t env_offset,
                      const uint32_t* tick_dev, void* stream);
int fg_random_actions_f64(void* act, int E, int N, uint64_t seed, uint32_t tick,
                          uint32_t env_offset, const uint32_t* tick_dev, void* stream);

/* The reference's hand-written controller for formation_hd_env, for every env of a batch in one launch:
 * get_action_BFS(ezpolicy, obs_n, num_agents_per_layer) (formation_gym/__init__.py:19-47,49-98; the default
 * policy of the reference's demo loop, test.py:23).  Works from the env STATE -- every value the reference
 * slices out of the per-agent observations is pos[b] - pos[a], ideal_shape or ideal_vel
 * (formation_hd_env.py:52-59) -- and writes act [E,N,2], ready for fg_step_fused.  N must be a power of
 * num_agents_per_layer (2..8), as the reference asserts (:55-56); unlike the reference, N = 243 with
 * 3 agents per layer is accepted (its floating-point log ratio 4.999999999999999 fails that assertion). */
int fg_policy_bfs(const void* pos, const void* ideal_shape, const void* ideal_vel, void* act, int E, int N,
                  int num_agents_per_layer, void* stream);
int fg_policy_bfs_f64(const void* pos, const void* ideal_shape, const void* ideal_vel, void* act, int E, int N,
                      int num_agents_per_layer, void* stream);

/* The reference's demo loop in one call per step (test.py:14-28 without -r):
 *     act_n = get_action_BFS(ezpolicy, obs_n, n);  obs_n, reward_n, done_n, _ = env.step(act_n)
 * with the state on the device: n_steps times { fg_step_fused on b->act (random_actions = 0); b->act =
 * fg_policy_bfs(new state) }.  b->act [E,N,2] is read AND written: on entry it holds the actions of the first step
 * (fg_policy_bfs of the current state), on return those for the step after the last one -- computed from the state
 * the returned observations describe, i.e. the reset state for an env whose episode just ended (auto_reset).
 * formation_hd_env with silent agents only.  Where the warp-autonomous step kernel has an instantiation with the
 * controller compiled in -- uniform agents, no walls, landmarks not tracked, (N, n) in {(3,3), (4,2), (8,2), (16,4)},
 * the shapes for which one kernel was measured faster than two; fp32: the standard buffer set of fg_step_fused (step/done/indiv/ep_return/ep_collisions/stats
 * present, no comm) -- a step is ONE launch and the controller never re-reads the state from HBM; everything else
 * runs the two kernels above per step, with the same results (same device functions). */
int fg_step_policy(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L, int n_steps,
                   int num_agents_per_layer, int auto_reset, uint64_t seed, uint32_t tick, uint32_t env_offset,
                   void* stream);
int fg_step_policy_f64(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L, int n_steps,
                       int num_agents_per_layer, int auto_reset, uint64_t seed, uint32_t tick, uint32_t env_offset,
                       void* stream);
/* fg_step_policy whose auto-resets take the env's task from a target bank (fg_targets, see fg_reset_targets); the
 * controller then steers towards the new task from the first step of the episode.  Same dispatch (one launch or two
 * per step) as fg_step_policy. */
int fg_step_policy_targets(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L, int n_steps,
                           int num_agents_per_layer, int auto_reset, uint64_t seed, uint32_t tick,
                           uint32_t env_offset, void* stream, const fg_targets* t);
int fg_step_policy_targets_f64(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L,
                               int n_steps, int num_agents_per_layer, int auto_reset, uint64_t seed, uint32_t tick,
                               uint32_t env_offset, void* stream, const fg_targets* t);

/* fg_step_fused_targets / fg_step_policy_targets that also record the terminal state of every env whose episode ends
 * in this call into the terminal block f (fg_final above).  f == NULL is exactly the _targets call; t == NULL is
 * allowed (no bank).  Everything the call computes -- obs, reward, done, indiv, state, step, episode statistics,
 * nan_flag, the Philox draws -- is bit for bit the call without a block.  FG_ERR_ARG, before any device call, when
 * f != NULL and: auto_reset == 0 or n_steps != 1; pos or vel is NULL; formation_hd_env lacks ideal_shape or
 * ideal_vel; another scenario lacks landmarks; non-silent agents lack comm; a pointer is not 8-byte (fp32) /
 * 16-byte (fp64) aligned.  The target-bank checks are those of the _targets calls. */
int fg_step_fused_final(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L,
                        int n_steps, int random_actions, int auto_reset, uint64_t seed, uint32_t tick,
                        uint32_t env_offset, void* stream, const fg_targets* t, const fg_final* f);
int fg_step_fused_final_f64(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L,
                            int n_steps, int random_actions, int auto_reset, uint64_t seed, uint32_t tick,
                            uint32_t env_offset, void* stream, const fg_targets* t, const fg_final* f);
int fg_step_policy_final(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L, int n_steps,
                         int num_agents_per_layer, int auto_reset, uint64_t seed, uint32_t tick,
                         uint32_t env_offset, void* stream, const fg_targets* t, const fg_final* f);
int fg_step_policy_final_f64(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L,
                             int n_steps, int num_agents_per_layer, int auto_reset, uint64_t seed, uint32_t tick,
                             uint32_t env_offset, void* stream, const fg_targets* t, const fg_final* f);

/* Terminal observations: obs [E,N,D] rows of every env with done[e*N] != 0, computed from the terminal block f by the
 * observation code of fg_obs_reward -- bit-identical to the rows the same step writes with auto_reset == 0.  Rows of
 * other envs are unspecified (a CTA holding an ended env also rewrites its other envs' rows).  Writes no other memory:
 * no reward, no landmark side effect, no nan_flag.  A CTA whose envs all have done == 0 exits before any observation
 * work, so a call after a step where no episode ended costs about one launch.  Same FG_ERR_ARG rules for f as the
 * _final steps (without the auto_reset / n_steps ones); done and obs must be non-null. */
int fg_final_obs(const fg_params* p, const fg_final* f, const uint8_t* done, void* obs, int scenario, int E, int N,
                 int L, void* stream);
int fg_final_obs_f64(const fg_params* p, const fg_final* f, const uint8_t* done, void* obs, int scenario, int E, int N,
                     int L, void* stream);

/* Observations of sampled state records (a replay buffer that stores states, not observations).  `states` is a block of
 * R records laid out like a terminal block with R in place of E: pos / vel / comm (non-silent agents) [R,N,2], and
 * ideal_shape [R,N,2] + ideal_vel [R,2] (formation_hd_env) or landmarks [R,L,2] (every other scenario;
 * formation_hd_obs_env: goals, then obstacles).  rows: DEVICE int64 [B].  obs [B,N,D]: slot b gets the observation rows
 * of record rows[b], computed by the observation code of fg_obs_reward -- bit-identical to what fg_obs_reward writes for
 * that state, which is what the step returned when the state was current.  Indices may repeat and come in any order;
 * records are addressed in 64 bits.  An index outside [0, R), negative included, reads nothing and gives slot b a row
 * block of NaN.  Writes no other memory: no reward, no landmark side effect, no nan_flag.  FG_ERR_ARG, before any
 * device call, when states, rows or obs is NULL, R < 1 or B < 1, or on the block rules of fg_final_obs (missing or
 * misaligned arrays); rows must be 8-byte aligned. */
int fg_obs_gather(const fg_params* p, const fg_final* states, long long R, const int64_t* rows, int B, void* obs,
                  int scenario, int N, int L, void* stream);
int fg_obs_gather_f64(const fg_params* p, const fg_final* states, long long R, const int64_t* rows, int B, void* obs,
                      int scenario, int N, int L, void* stream);

/* Prioritized replay over the transitions of a state-record replay buffer of `slots` slots x `envs` envs (proportional
 * PER, Schaul et al. 2016, as in baselines' PrioritizedReplayBuffer): a 32-ary sum tree with a min per node.
 *   Leaves: leaf[j*envs + e] > 0 (the priority) exactly when slot j, env e holds a transition; 0 otherwise.  M = slots *
 *   envs <= 2^40.  Level 0 is the leaves, read as padded with zeros to a multiple of 32; node i of level k+1 reduces
 *   nodes 32i .. 32i+31 of level k (children past the end of a level count as sum 0 / min +inf); levels 1 .. depth are
 *   stored in `sum` / `min` bottom level first, the root (one node) last.  sum = the butterfly sum of the 32 children
 *   (v_l = v_l + v_{l^off} for off = 16, 8, 4, 2, 1, then v_0: a __shfl_xor reduction); min = the minimum over the
 *   nonzero leaves below, +inf for none.  The tree is a pure function of the leaves.
 *   Caller-owned device memory, sized by fg_per_layout and initialised ONCE to: leaf 0, sum 0, min +inf, max_leaf 1.0,
 *   stamp 0, prev -1, scratch 0 (the calls leave scratch 0 again).  Arrays 8-byte aligned, scratch 4-byte.
 * None of the calls allocates or synchronises; every argument error returns FG_ERR_ARG before any device call. */
typedef struct fg_per {
    double* leaf;              /* [slots*envs] */
    double* sum;               /* [nodes] internal nodes of every level, bottom level first, root last */
    double* min;               /* [nodes] same layout */
    double* max_leaf;          /* [1] running maximum of the leaf values fg_per_update wrote (initially 1.0) */
    int64_t* stamp;            /* [slots] write count of each slot (fg_per_fill) */
    int64_t* prev;             /* [slots] slot holding the s of slot j's transition, -1 for none */
    void* scratch;             /* [scratch_bytes] duplicate resolution of fg_per_update */
    long long slots, envs;
} fg_per;

/* Sizes of the tree of slots x envs leaves: internal nodes (all levels), depth (levels above the leaves, >= 1) and the
 * scratch bytes.  FG_ERR_ARG when a pointer is NULL, slots or envs < 1, or slots * envs > 2^40.  Host only. */
int fg_per_layout(long long slots, long long envs, long long* nodes, int* depth, long long* scratch_bytes);
/* A slot was written: stamp[slot] = stamp, prev[slot] = prev, the leaves of `slot` = *max_leaf when valid (a transition:
 * prev >= 0) else 0 (a chain start), the leaves of drop_slot (-1: none; the transition whose s `slot` held) = 0, then
 * their ancestors.  FG_ERR_ARG unless 0 <= slot < slots, prev and drop_slot are -1 or another slot, valid is 0 / 1,
 * stamp >= 0. */
int fg_per_fill(const fg_per* t, long long slot, long long prev, long long stamp, int valid, long long drop_slot,
                void* stream);
/* Priority update for B sampled transitions: index [B] (leaf), stamp [B] (the slot stamp fg_per_sample returned), td [B]
 * (fp32, or fp64 when td_f64 = 1; device).  Entry b is applied when td[b] is finite, 0 <= index[b] < M, the leaf is > 0
 * and stamp[slot] still equals stamp[b]; among applied entries of one leaf the largest b wins.  The leaf becomes
 * clamp((|td| + eps)^alpha, 2^-1022, 2^960), max_leaf the max of itself and the values written, then the ancestors are
 * recomputed.  FG_ERR_ARG also when B < 1, alpha < 0, eps <= 0 or either is not finite. */
int fg_per_update(const fg_per* t, const int64_t* index, const int64_t* stamp, const void* td, int td_f64, int B,
                  double alpha, double eps, void* stream);
/* B proportional draws: u [B] fp64 in [0, 1) (device), x = u * root.sum; from the root take the smallest child k with
 * c_k > 0 and x < P_k (inclusive prefix sum), else the last child with c_k > 0, then x -= P_{k-1} clamped into [0, c_k).
 * A zero leaf is never returned.  Per draw b, with leaf l = slot * envs + e: rows[b] = prev[slot] * envs + e and
 * rows[B + b] = l + (done[l] ? M : 0) (the record rows of s and s' in StateReplayBuffer's block, for fg_obs_gather),
 * index[b] = l, stamp_out[b] = stamp[slot], slot_out[b], env_out[b], done_out[b] = done[l], weights[b] =
 * (root.min / leaf)^beta (fp64, stored in the real type), actions_out [B,N,A] = actions[l] and reward_out [B,N] =
 * reward[l] from done [slots*envs] (uint8), actions [slots*envs,N,A] and reward [slots*envs,N].  An empty tree gives
 * -1 indices and NaN.  FG_ERR_ARG also when B < 1, N outside [1, FG_MAX_AGENTS], A outside [1, 64], beta < 0 or not
 * finite, a pointer NULL or not aligned to its type. */
int fg_per_sample(const fg_per* t, const double* u, int B, double beta, const uint8_t* done, const void* actions,
                  const void* reward, int N, int A, int64_t* rows, int64_t* index, int64_t* stamp_out,
                  int64_t* slot_out, int64_t* env_out, uint8_t* done_out, void* weights, void* actions_out,
                  void* reward_out, void* stream);
int fg_per_sample_f64(const fg_per* t, const double* u, int B, double beta, const uint8_t* done, const void* actions,
                      const void* reward, int N, int A, int64_t* rows, int64_t* index, int64_t* stamp_out,
                      int64_t* slot_out, int64_t* env_out, uint8_t* done_out, void* weights, void* actions_out,
                      void* reward_out, void* stream);

/* Generalized advantage estimation (Schulman et al. 2016) over an on-policy rollout of T steps of E envs x N agents,
 * with time-limit truncations bootstrapped from the value of the state the episode ended in.  M = E*N columns, column
 * c = e*N + n; all arrays on the device, in the real type (fp32 / fp64 for _f64) except done:
 *   reward [T,E,N]; value [T+1,E,N]: value[t] = V(s_t), value[T] the bootstrap value of the rollout's last state;
 *   done [T,E] uint8: nonzero when env e's episode ended at step t (env.done[:, 0]);
 *   final_value [T,E,N] or NULL: V of the state the episode that ended at step t ended in; read only where done[t,e];
 *   adv, ret [T,E,N]: outputs.
 * With g = (real)gamma and gl = (real)(gamma * lambda) (the product taken in fp64 and rounded once), for every column
 * from a = 0 and t = T-1 .. 0, every operation separately rounded (no contraction, in both precisions):
 *   d = done[t*E + e] != 0;  nv = d ? (final_value ? final_value[t*M + c] : 0) : value[(t+1)*M + c]
 *   delta = (reward[t*M + c] + g*nv) - value[t*M + c];  a = d ? delta : delta + gl*a
 *   adv[t*M + c] = a;  ret[t*M + c] = a + value[t*M + c]
 * final_value == NULL treats a truncation as a terminal.  value[t+1] after a done is never read into the result, so a
 * NaN or inf there does not reach adv / ret.  Every column is independent: the result does not depend on the launch
 * geometry.  No allocation, no synchronisation.  FG_ERR_ARG, before any device call, when reward / value / done / adv /
 * ret is NULL, T < 1, E < 1, N outside [1, FG_MAX_AGENTS], T*E*N > 2^48, gamma or lambda is not finite or outside
 * [0, 1], or an array is not aligned to the real type. */
int fg_gae(const void* reward, const void* value, const void* final_value, const uint8_t* done, void* adv, void* ret,
           int T, long long E, int N, double gamma, double lambda, void* stream);
int fg_gae_f64(const void* reward, const void* value, const void* final_value, const uint8_t* done, void* adv,
               void* ret, int T, long long E, int N, double gamma, double lambda, void* stream);

/* Diagnostics, not on the step path: FP32 pipe probes used by bench.py to MEASURE the FP32 peak the
 * large-N step+reward kernel is graded against (BASELINE.json north_star: "% of FP32 peak at 243
 * agents"; MEASURED_PEAKS.json holds no FP32 figure).  variant 0: scalar FFMA (2 flop/lane/instr),
 * 1: packed FFMA2 (fma.rn.f32x2; 4 flop/lane/instr), 2: FMNMX (1 op), 3: the pair-loop instruction mix
 * (FADD2, FADD2, FMUL2, FFMA2, FMNMX3 per two pairs).  Each of ctas x 256 threads runs `iters`
 * iterations of 32 instructions (variants 0-2) or 8 pair-steps of 7 instructions (variant 3);
 * `scratch` is a device buffer of >= ctas*256 floats (never written in practice).  Time it with
 * CUDA events on `stream`. */
int fg_fp32_probe(int variant, int iters, int ctas, float* scratch, void* stream);

/* Diagnostics: write-only HBM stream over `bytes` of `dst` (what an observation writer can reach at
 * best).  variant 0: 16-byte streaming stores; 1: TMA bulk stores (cp.async.bulk) of `chunk` bytes from
 * shared memory; 2: the same with the L2 evict_first policy the step kernels use; 4: as 2, each CTA writing its own
 * contiguous range of chunks instead of chunks b, b + ctas, ...; 3: hd observation rows of
 * `chunk` = N agents written with plain 8-byte streaming stores from registers (one warp per env, 128-thread CTAs). */
int fg_write_probe(int variant, void* dst, unsigned long long bytes, unsigned chunk, int ctas, void* stream);

/* VecEnv adapter, host side of the boundary (train/maddpg-v2/utils/env_wrappers.py:68-72: the trainers read
 * obs[E,N,D] as a HOST array after every step): ship one step's observation tensor from `obs_dev` [E*N rows x
 * row_items items of item_bytes (8 = float2, 16 = double2)] into the pinned, persistent host array `obs_host` of the
 * same layout.  Only the first `dyn_items` items of a row change every step (hd: [p_vel | other_pos] = N of 3N items,
 * formation_hd_env.py:52-59); the rest changes when the env is reset, so a step needs a third of the PCIe bytes to
 * leave the host array byte-identical to the device tensor.
 *   mode 0: whole tensor, one contiguous copy.
 *   mode 1: 2-D copy-engine transfer of the dynamic prefix of every row (the caller uses mode 0 on steps that
 *           reset envs).
 *   mode 2: scatter kernel storing straight into the mapped pinned host array: dynamic prefix of every row, WHOLE
 *           rows where done_dev[row] != 0 (done [E,N] uint8 of the same step; NULL = no whole rows).
 *   mode 3: pack the dynamic prefixes into `staging_dev` [E*N, dyn_items], then one contiguous copy of that into
 *           `obs_host` (which then is a [E*N, dyn_items] staging array; diagnostic).
 *   mode 4: as 2, but in whole 64-byte host cache lines (the lines a row's dynamic prefix -- or, where done_dev says so,
 *           the whole row -- touches; the extra bytes are row items whose host copy already equals the device value).
 *           obs_dev / obs_host 64-byte aligned, E*N*row_items*item_bytes a multiple of 16, else FG_ERR_ARG.
 * Asynchronous on `stream`; the caller synchronises before reading the host array. */
int fg_obs_to_host(const void* obs_dev, void* obs_host, const uint8_t* done_dev, void* staging_dev, int E, int N,
                   int row_items, int dyn_items, int item_bytes, int mode, void* stream);

/* Launch geometry chosen for (N): envs per CTA and threads per CTA (for reporting/tests). */
int fg_launch_geometry(int N, int* envs_per_cta, int* threads_per_cta);

#ifdef __cplusplus
}
#endif
#endif /* FORMATION_GYM_B200_H */

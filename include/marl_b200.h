/* marl_b200.h — C-ABI of the B200-native MAPPO rollout-and-update hot path.
 *
 * The reference (Desperodoo/distributed_multi_agent_reinforcement_learning) is pure Python and has no FFI
 * of its own; its plugin surface is Python duck typing resolved by hydra `_target_` strings
 * (config.yaml:14-15,56-57; runner.py:19,84-85).  This header is the boundary a maintainer binds with
 * ctypes (see INTEGRATION.md): every entry point below replaces the body of one reference method and is
 * cited with the reference file:line it replaces.
 *
 * Conventions (all entry points):
 *   - plain C, `extern "C"`, raw pointers + explicit sizes; no torch / C++ types cross the boundary;
 *   - every pointer named d_* is a DEVICE pointer (HBM) owned by the caller; the library never allocates,
 *     frees or synchronises; `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - returns 0 (MARL_OK) or a negative MARL_E* code; never throws, never exits;
 *     marl_last_error_string() describes the most recent failure on the calling thread;
 *   - no global mutable state besides that thread-local error string: re-entrant, one host thread per GPU.
 *
 * Layouts (row-major, "pursuer" == reference "defender", "evader" == reference "attacker"):
 *   p_state   f64 [B,N,4]   (x,y,vx,vy)             base_env.py:198-209, pursuit_env.py:179-180
 *   e_state   f64 [B,4]
 *   grid bits u32 [M,W,HW]  HW=ceil(H/32); bit (y&31) of word [m,x,y>>5] == occupied_map.grid_map[x][y]
 *   raser     u32 [M,W*H,OW] OW=ceil(O/32); bit k of row (x*H+y) == raser_map[x][y][k]  pursuit_env.py:29-53
 *   map_id    i32 [B]       env b uses map map_id[b] of the pool (NULL => map b)
 */
#ifndef MARL_B200_H
#define MARL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MARL_ABI_VERSION 1

enum {
    MARL_OK = 0,
    MARL_EINVAL = -1,     /* bad argument (null pointer, size out of the supported range) */
    MARL_ECUDA = -2,      /* a CUDA runtime call / kernel launch failed */
    MARL_EUNSUPPORTED = -3
};

#define MARL_MAX_AGENTS 128   /* N <= 128 (one warp per env, up to 4 pursuers per lane) */
#define MARL_NUM_ACTIONS 9    /* agent.py:57-60: 8 headings + stop */

/* Scalar configuration of one Pursuit_Env family (config.yaml:13-54 / conf/{env,attacker,defender,sensor,mao}.yaml). */
typedef struct marl_env_params {
    int32_t W, H;              /* map.map_size */
    int32_t N;                 /* env.num_defender */
    int32_t O;                 /* map.num_max_obstacle: padded width of every obstacle-adjacency row */
    int32_t max_steps;         /* env.max_steps */
    int32_t difficulty;        /* env.difficulty: evader replans every `difficulty` steps */
    int32_t sensor_beams;      /* sensor.num_beams */
    int32_t sensor_radius;     /* sensor.radius */
    int32_t e_extend_dis;      /* attacker.extend_dis */
    int32_t e_sen_range;       /* attacker.sen_range (window of Evader.rescan) */
    double d_step, d_tau, d_vmax, d_collision_radius, d_comm_range, d_sen_range;   /* defender.* */
    double e_step, e_tau, e_vmax, e_collision_radius;                               /* attacker.* */
    double resolution;         /* map.resolution */
} marl_env_params;

int marl_version(void);
const char *marl_last_error_string(void);

/* ---- kernel 1: batched pursuer step --------------------------------------------------------------
 * Replaces Pursuit_Env.step + defender_reward + collision_detection + Agent.step/dynamic
 * (environment/pursuit_evasion_game/pursuit_env.py:104-177, agent.py:62-104, Occupied_Grid_Map.py:65-115).
 * d_action_table f64 [9,2] is Agent.actions_mat (agent.py:57-60) computed by the caller with numpy so that
 * cos/sin come from the same libm the reference would use.
 * In/out: d_p_state, d_time_step (i32 [B], += 1), d_collision (u8 [B], sticky OR of any rejected move).
 * Out: d_reward i32 [B,N], d_can_apply u8 [B,N], d_done u8 [B] (time_step >= max_steps). */
int marl_env_step(const marl_env_params *p, int32_t B, int32_t M,
                  double *d_p_state, const double *d_e_state, const int32_t *d_action,
                  const uint32_t *d_grid_bits, const int32_t *d_map_id, const double *d_action_table,
                  int32_t *d_reward, uint8_t *d_can_apply, uint8_t *d_collision, int32_t *d_time_step,
                  uint8_t *d_done, void *stream);

/* ---- kernel 2: observations ----------------------------------------------------------------------
 * Replaces Pursuit_Env.communicate (pursuit_env.py:182-195, including the `adj_mat[j, 1] = 1` quirk) and
 * Pursuit_Env.sensor + Pursuer.find_attacker + bresenham_line (pursuit_env.py:197-209, agent.py:157-169,319-341).
 * Packed outputs (canonical): d_p_adj_bits u32 [B,N,NW] NW=ceil(N/32); d_e_adj u8 [B,N]; d_o_adj_bits u32 [B,N,OW].
 * Dense outputs (reference ReplayBuffer layout, any may be NULL): d_p_adj_f32 [B,N,N], d_e_adj_f32 [B,N,1],
 * d_o_adj_f32 [B,N,O]. */
int marl_env_observe(const marl_env_params *p, int32_t B, int32_t M,
                     const double *d_p_state, const double *d_e_state,
                     const uint32_t *d_grid_bits, const uint32_t *d_raser_bits, const int32_t *d_map_id,
                     uint32_t *d_p_adj_bits, uint8_t *d_e_adj, uint32_t *d_o_adj_bits,
                     float *d_p_adj_f32, float *d_e_adj_f32, float *d_o_adj_f32, void *stream);

/* ---- kernel 2b: per-map sensor tables ------------------------------------------------------------
 * Replaces get_boundary_map + get_raser_map (pursuit_env.py:18-53; find_boundaries(mode='inner') is
 * scikit-image 0.19.3, restated).  d_beam_dir f64 [beams,2] = (cos,sin)(beam*2*pi/beams) from the caller's numpy.
 * Out: d_boundary_bits u32 [M,W,HW]; d_boundary_count i32 [M]; d_boundary_xy i32 [M,O,2] (np.argwhere order,
 * rows >= count are zero); d_raser_bits u32 [M,W*H,OW].  A map with more than O boundary cells sets
 * count to the true number and truncates the list (the reference would raise on buffer store). */
int marl_raser_map_build(const marl_env_params *p, int32_t M, const uint32_t *d_grid_bits,
                         const double *d_beam_dir, uint32_t *d_boundary_bits, int32_t *d_boundary_count,
                         int32_t *d_boundary_xy, uint32_t *d_raser_bits, void *stream);

/* ---- kernel 1c: evader (A* replanning + waypoint following) --------------------------------------
 * Replaces Pursuit_Env.attacker_step + Evader.{replan,rescan,waypoint2phi,step} + AStar_2D.searching
 * (pursuit_env.py:75-102, agent.py:197-271, astar.py:26-161, Occupied_Grid_Map.py:119-191).
 * One call == one attacker_step for B envs.  State per env: d_e_state f64 [B,4] (in/out), d_target i32 [B,2]
 * (in/out), d_path i16 [B,path_cap,2] + d_path_len i32 [B] (in/out; path[len-1] is the next waypoint, as in the
 * reference list), d_time_step i32 [B] (read: replan iff time_step % difficulty == 0).
 * Target resampling (base_env.py:52-70 via pursuit_env.py:98-100) consumes candidates from
 * d_target_tape i32 [B,tape_len,2] at cursor d_tape_pos i32 [B] (in/out): candidates occupied in the
 * 2-inflated map are skipped exactly like the rejection loop.  d_inflated_bits u32 [M,W,HW].
 * d_status i32 [B] (may be NULL) is OR-ed with MARL_EV_* bits; a non-zero status means the result for that env
 * is NOT the reference's (search heap or path buffer overflow, tape exhausted) and must be treated as an error.
 * d_e_tape2 f64 [2,B,4] (may be NULL) receives the evader state before ([0]) and after ([1]) this step — the
 * 2-slot tape marl_rollout_steps(K=1) consumes, so a closed-loop env step is two launches.
 * Supported maps: H <= 63, W <= 254 (one 64-bit column per x in shared memory). */
#define MARL_EV_HEAP_OVERFLOW 1
#define MARL_EV_PATH_OVERFLOW 2
#define MARL_EV_TAPE_EXHAUSTED 4
#define MARL_EV_MISSED_REPLAN 8   /* marl_rollout_closed stepped across a replanning boundary */
int marl_evader_step(const marl_env_params *p, int32_t B, int32_t M,
                     double *d_e_state, const double *d_p_state, int32_t *d_target,
                     int16_t *d_path, int32_t *d_path_len, int32_t path_cap,
                     const int32_t *d_time_step,
                     const uint32_t *d_grid_bits, const uint32_t *d_inflated_bits, const int32_t *d_map_id,
                     const int32_t *d_target_tape, int32_t tape_len, int32_t *d_tape_pos,
                     int32_t *d_status, double *d_e_tape2, void *stream);

/* Replanning only (Evader.replan, agent.py:232-259) for the envs with time_step % difficulty == 0; the others
 * return immediately.  Used by the chunked closed-loop rollout: one replan launch per `difficulty` steps, the
 * per-step move being fused into marl_rollout_closed. */
int marl_evader_replan(const marl_env_params *p, int32_t B, int32_t M, const double *d_e_state,
                       const double *d_p_state, const int32_t *d_target, int16_t *d_path, int32_t *d_path_len,
                       int32_t path_cap, const int32_t *d_time_step, const uint32_t *d_grid_bits,
                       const int32_t *d_map_id, int32_t *d_status, void *stream);

/* ---- episode initialisation on the device -----------------------------------------------------------------------------------
 * Replaces Pursuit_Env.reset's generators for large batches (pursuit_env.py:60-73 -> base_env.py:37-162, Occupied_Grid_Map.py:46-62).
 * Same placement RULES as the reference (blocks of 6x6 cells around N(center, variance); target on a free cell of the 2-inflated
 * map; every pursuer on a free cell, >= min_dist from the earlier ones and within comm range of one or two of them, its
 * `extend`-inflated footprint then blocked; evader on a free point within sen_range of a pursuer cell), but every map / env draws
 * from its own counter-based stream keyed by (seed, index): rule- and distribution-equivalent, not stream-equivalent — the
 * single-env facade keeps the reference's global-RNG order on the host (maps.py).
 * marl_map_generate: d_grid_bits, d_inflated_bits u32 [M,W,HW] out.
 * marl_env_reset_place: d_p_state f64 [B,N,4], d_e_state f64 [B,4], d_target i32 [B,2] out (velocities zero); d_scratch u32
 * [B,W,HW]; d_fail i32 [B] (may be NULL) is 1 where more than max_draws proposals were rejected (over-crowded map). */
int marl_map_generate(const marl_env_params *p, int32_t M, int32_t num_blocks, double center_x, double center_y, double variance,
                      uint64_t seed, uint32_t *d_grid_bits, uint32_t *d_inflated_bits, void *stream);
int marl_env_reset_place(const marl_env_params *p, int32_t B, int32_t M, const uint32_t *d_inflated_bits, const int32_t *d_map_id,
                         uint64_t seed, double min_dist, int32_t extend, int32_t max_draws, double *d_p_state, double *d_e_state,
                         int32_t *d_target, uint32_t *d_scratch, int32_t *d_fail, void *stream);

/* ---- kernel 3a: Welford reward normalisation -----------------------------------------------------
 * Replaces Normalization.__call__ / RunningMeanStd.update (DHGN/normalization.py:4-35) applied per env:
 * d_n i64 [B], d_mean f64 [B,N], d_S f64 [B,N], d_std f64 [B,N] (in/out); d_reward i32 [B,N] in;
 * d_out f32 [B,N] = float32((x-mean)/(std+1e-8)) (DHGN/mappo_parallel.py:795-797). update != 0 => update stats. */
int marl_welford_update(int32_t B, int32_t N, const int32_t *d_reward, int64_t *d_n, double *d_mean,
                        double *d_S, double *d_std, float *d_out, int32_t update, void *stream);
/* Same estimate fed with f64 samples d_x [B,N]: RunningMeanStd.update on the discounted return of RewardScaling
 * (DHGN/normalization.py:38-52), whose samples are not integers. */
int marl_welford_update_f64(int32_t B, int32_t N, const double *d_x, int64_t *d_n, double *d_mean,
                            double *d_S, double *d_std, float *d_out, int32_t update, void *stream);

/* ---- kernel 3b: GAE + advantage normalisation ----------------------------------------------------
 * Replaces MAPPO.train's GAE block (DHGN/mappo_parallel.py:643-658).  time_major == 0: r, active f32 [B,T,N],
 * v f32 [B,T+1,N] (reference ReplayBuffer layout); time_major != 0: [T,B,N] / [T+1,B,N] (rollout arena layout).
 * Out: adv, v_target in the same layout as r.  gamma_lamda = float32(gamma*lamda) with the product taken in
 * double, as Python does.  If use_adv_norm, adv = (adv-mean)/(std_unbiased+1e-5)*active over the whole tensor.
 * d_workspace: >= marl_gae_workspace_bytes(B,T,N) bytes. */
int64_t marl_gae_workspace_bytes(int32_t B, int32_t T, int32_t N);
int marl_gae(int32_t B, int32_t T, int32_t N, const float *d_r, const float *d_v, const float *d_active,
             int32_t time_major, float gamma, float gamma_lamda, int32_t use_adv_norm, float *d_adv,
             float *d_v_target, void *d_workspace, void *stream);

/* ---- kernel 4: minibatch gather ------------------------------------------------------------------
 * Replaces `batch[key][index]` (DHGN/mappo_parallel.py:665-679): copies rows d_index[i] (i < n_index) of a
 * [B,row_bytes] byte matrix into [n_index,row_bytes].  row_bytes must be a multiple of 4; 16-byte aligned
 * rows take the vectorised path. */
int marl_gather_rows(const void *d_src, void *d_dst, const int64_t *d_index, int32_t n_index,
                     int64_t row_bytes, int64_t n_src_rows, void *stream);

/* ---- fused rollout (env-only hot loop with a device-side action source) --------------------------
 * K consecutive iterations of the reference rollout body (DHGN/mappo_parallel.py:758-801) without the
 * network: observe -> [evader tape] -> step -> reward-norm -> store.  Actions come from d_action_tape
 * i32 [K,B,N] or, when NULL, from a counter-based uniform{0..8} generator seeded by `seed` (throughput runs).
 * Evader states come from d_e_tape f64 [K+1,B,4] (state before each iteration's attacker_step at [k], after at
 * [k+1]).  Records for iteration k land at time index t0+k of the TIME-MAJOR rollout arena (DESIGN.md §3; the
 * reference's [B,T,...] tensors are zero-copy permuted views of it).  Any record pointer may be NULL.
 * Generated actions: uniform{0..8} = ((splitmix64(seed ^ splitmix64(agent*0x100000001B3 + t)) >> 32) * 9) >> 32
 * with agent = b*N+i and t = t0+k. */
typedef struct marl_rollout_records {   /* all TIME-MAJOR: one step of all envs is one contiguous slab */
    float *p_state_f32;        /* [T,B,N,4]  float32(p_state before the step)  replay_buffer.py:47 */
    float *e_state_f32;        /* [T,B,1,4]                                    replay_buffer.py:48 */
    uint32_t *p_adj_bits;      /* [T,B,N,NW] */
    uint8_t *e_adj;            /* [T,B,N]    */
    uint32_t *o_adj_bits;      /* [T,B,N,OW] */
    float *a_n;                /* [T,B,N]    float32(action)                   replay_buffer.py:57 */
    float *r;                  /* [T,B,N]    normalised reward                 replay_buffer.py:59 */
    int32_t *raw_reward;       /* [T,B,N]    un-normalised integer reward */
    float *active;             /* [T,B,N]    always 1                          mappo_parallel.py:798 */
    float *p_adj_f32;          /* [T,B,N,N]  dense fp32 as the reference stores it (optional) replay_buffer.py:50 */
    float *e_adj_f32;          /* [T,B,N,1] */
    float *o_adj_f32;          /* [T,B,N,O] */
} marl_rollout_records;

int marl_rollout_steps(const marl_env_params *p, int32_t B, int32_t M, int32_t T, int32_t t0, int32_t K,
                       double *d_p_state, const double *d_e_tape, const int32_t *d_action_tape, uint64_t seed,
                       const uint32_t *d_grid_bits, const uint32_t *d_raser_bits, const int32_t *d_map_id,
                       const double *d_action_table,
                       int64_t *d_wf_n, double *d_wf_mean, double *d_wf_S, double *d_wf_std,
                       uint8_t *d_collision, int32_t *d_time_step,
                       const marl_rollout_records *rec, void *stream);

/* Closed-loop variant: the evader is simulated on the device.  K <= difficulty consecutive iterations of
 * observe -> attacker_step's move (waypoint following, dynamics, target resampling from the tape) -> step ->
 * reward-norm -> store; the caller launches marl_evader_replan before every chunk that starts on a replanning
 * boundary (time_step % difficulty == 0).  Evader state arguments as in marl_evader_step.
 * Sub-batches: to roll envs [e0, e0+B) of an arena holding B_stride envs per time slab, pass every per-env pointer
 * (record and action-tape pointers included) already offset to env e0, B_stride = the arena's env count (0 means B)
 * and env0 = e0 (it keys the action generator so that sub-batching does not change the actions).  Independent
 * sub-batches can then run on different streams, so one slow A* search only delays its own sub-batch. */
int marl_rollout_closed(const marl_env_params *p, int32_t B, int32_t B_stride, int32_t env0, int32_t M, int32_t T, int32_t t0,
                        int32_t K, double *d_p_state, double *d_e_state, int32_t *d_target, const int16_t *d_path,
                        int32_t *d_path_len, int32_t path_cap, const uint32_t *d_inflated_bits,
                        const int32_t *d_target_tape, int32_t tape_len, int32_t *d_tape_pos,
                        int32_t *d_evader_status, const int32_t *d_action_tape, uint64_t seed,
                        const uint32_t *d_grid_bits, const uint32_t *d_raser_bits, const int32_t *d_map_id,
                        const double *d_action_table,
                        int64_t *d_wf_n, double *d_wf_mean, double *d_wf_S, double *d_wf_std,
                        uint8_t *d_collision, int32_t *d_time_step,
                        const marl_rollout_records *rec, void *stream);

/* ---- 3-D particle env (second env family, BASELINE config 4) --------------------------------------------
 * Replaces environment/env_3d/particle_env.py: Point.step (:25-57), ParticleEnv.step (:204-217),
 * reward / agent_reward (:263-279), update_agent_active (:281-321), get_done (:219-238), get_active (:240-244),
 * get_adj_mat (:323-334), collision_detection (:336-346) and the evader's Point.step inside evader_step (:348-373;
 * the commanded action itself comes from scipy SLSQP in eva.e_f and is an INPUT here).
 * Layouts: p_state f64 [B,N,6] (x,y,z,phi,gamma,v), p_active u8 [B,N], e_state f64 [B,6], e_active u8 [B],
 * target f64 [B,3], actions f64 in [-1,1]^3 (phi, gamma, v commands). */
typedef struct marl_env3d_params {
    int32_t N;                 /* p_num */
    int32_t max_step;          /* ParticleEnv.max_step (200) */
    double p_vmax, e_vmax;     /* 0.7 / 1 */
    double kill_radius;        /* 0.5 */
    double ang_lmt, v_lmt;     /* pi/4, 0.4 */
    double step_size;          /* 0.5 */
    double comm_range;         /* p_comm_range 6 (pursuer-pursuer adjacency) */
    double sen_range;          /* p_sen_range 3 (pursuer-evader adjacency) */
} marl_env3d_params;

/* One ParticleEnv.step for B envs: time_step += 1; every active pursuer moves; reward from the post-move state
 * (+1 per active evader within kill_radius, -(active teammates within kill_radius, self included, - 1)); pursuers /
 * the evader that touch anything are deactivated and parked at (1000,1000,1000,0,0,0); done = evader at target ||
 * no pursuer alive || evader dead || time_step >= max_step.  In/out: p_state, p_active, e_state, e_active,
 * time_step.  Out: reward i32 [B,N], done u8 [B]. */
int marl_env3d_step(const marl_env3d_params *p, int32_t B, double *d_p_state, uint8_t *d_p_active, double *d_e_state,
                    uint8_t *d_e_active, const double *d_target, const double *d_action, int32_t *d_time_step,
                    int32_t *d_reward, uint8_t *d_done, void *stream);
/* The evader's own Point.step (particle_env.py:372) for a commanded action d_e_action f64 [B,3]. */
int marl_env3d_evader_step(const marl_env3d_params *p, int32_t B, double *d_e_state, const uint8_t *d_e_active,
                           const double *d_e_action, void *stream);
/* get_adj_mat for the two relations a policy consumes: pursuer-pursuer within comm_range (rows of inactive pursuers
 * are zero; columns are not masked, as in the reference) and pursuer-evader within sen_range.
 * Out: d_pp_adj_bits u32 [B,N,NW], d_pe_adj u8 [B,N]; dense f32 [B,N,N] / [B,N,1] optional (NULL to skip). */
int marl_env3d_adjacency(const marl_env3d_params *p, int32_t B, const double *d_p_state, const uint8_t *d_p_active,
                         const double *d_e_state, uint32_t *d_pp_adj_bits, uint8_t *d_pe_adj, float *d_pp_adj_f32,
                         float *d_pe_adj_f32, void *stream);
/* K fused iterations of (adjacency -> evader move -> step -> store) with actions from tapes
 * (d_action_tape f64 [K,B,N,3], d_e_action_tape f64 [K,B,3]) or, when a tape is NULL, from the counter RNG
 * (uniform in [-1,1), keyed by seed / agent / t).  Time-major records (any may be NULL): p_state_f32 [T,B,N,6],
 * e_state_f32 [T,B,6], pp_adj_bits [T,B,N,NW], pe_adj u8 [T,B,N], reward i32 [T,B,N], active_f32 [T,B,N]
 * (active flag BEFORE the step, what a buffer stores), done u8 [T,B]. */
typedef struct marl_env3d_records {
    float *p_state_f32; float *e_state_f32; uint32_t *pp_adj_bits; uint8_t *pe_adj; int32_t *reward; float *active_f32;
    uint8_t *done;
} marl_env3d_records;
int marl_env3d_rollout(const marl_env3d_params *p, int32_t B, int32_t T, int32_t t0, int32_t K, double *d_p_state,
                       uint8_t *d_p_active, double *d_e_state, uint8_t *d_e_active, const double *d_target,
                       int32_t *d_time_step, const double *d_action_tape, const double *d_e_action_tape, uint64_t seed,
                       const marl_env3d_records *rec, void *stream);

/* ---- third env family: 2-D N-pursuers-vs-E-evaders particle env (environment/env_n2n/particle_env.py) ----------------------
 * State: pursuers f64 [B,N,4] = (x, y, phi, v), evaders f64 [B,E,4], active u8 [B,N] / [B,E], target f64 [B,2], time_step i32 [B].
 * N, E <= 32.  Pursuers take the discrete heading actions 0..8 (0 = stop), evaders a commanded heading in [-1,1] (the reference's
 * SLSQP evader `eva.e_f` is third-party arithmetic: its output is an input here).
 * marl_envn2n_step        = ParticleEnv.step (:164-177): Pursuer.step of every pursuer (an inactive one still turns, :34-63), reward
 *                           (:263-285), update_agent_active (:287-321, parked at (1000,1000), phi 0), get_done (:248-262) / episode_limit.
 * marl_envn2n_evader_step = the Evader.step half of evader_step (:179-193, :70-93) for commanded headings d_e_action f64 [B,E].
 * marl_envn2n_observe     = get_adj_mat (:338-350) for pursuer-pursuer (comm_range) and pursuer-evader (sen_range) as one word per
 *                           pursuer (bit j = column j; rows of inactive pursuers are zero) and choose_evader('actor') (:392-420) as the
 *                           index of the chosen evader or -1.
 * marl_envn2n_rollout     = K fused iterations of (observe -> evader move -> step -> store) with actions from tapes (d_action_tape i32
 *                           [K,B,N], d_e_action_tape f64 [K,B,E]) or, when a tape is NULL, from the counter RNG.  Time-major records
 *                           (any may be NULL): states / active flags BEFORE the step, observations, actions, rewards, done. */
typedef struct marl_envn2n_params {
    int32_t N, E;              /* p_num, e_num */
    int32_t episode_limit;     /* 100 */
    int32_t reserved;
    double p_vmax;             /* 0.3 (the evaders' speed is part of their state) */
    double kill_radius;        /* 0.5 */
    double ang_lmt;            /* pi/4 */
    double step_size;          /* 0.5 */
    double comm_range;         /* p_comm_range 6 */
    double sen_range;          /* p_sen_range 3 */
} marl_envn2n_params;
typedef struct marl_envn2n_records {
    float *p_state_f32;        /* [T,B,N,4] */
    float *e_state_f32;        /* [T,B,E,4] */
    uint8_t *p_active;         /* [T,B,N] */
    uint8_t *e_active;         /* [T,B,E] */
    uint32_t *pp_adj_bits;     /* [T,B,N] */
    uint32_t *pe_adj_bits;     /* [T,B,N] */
    int8_t *assign;            /* [T,B,N] */
    int32_t *action;           /* [T,B,N] */
    int32_t *reward;           /* [T,B,N] */
    uint8_t *done;             /* [T,B] */
} marl_envn2n_records;
int marl_envn2n_step(const marl_envn2n_params *p, int32_t B, double *d_p_state, uint8_t *d_p_active, double *d_e_state,
                     uint8_t *d_e_active, const double *d_target, const int32_t *d_action, int32_t *d_time_step,
                     int32_t *d_reward, uint8_t *d_done, void *stream);
int marl_envn2n_evader_step(const marl_envn2n_params *p, int32_t B, double *d_e_state, uint8_t *d_e_active,
                            const double *d_e_action, void *stream);
int marl_envn2n_observe(const marl_envn2n_params *p, int32_t B, const double *d_p_state, const uint8_t *d_p_active,
                        const double *d_e_state, const uint8_t *d_e_active, uint32_t *d_pp_adj_bits, uint32_t *d_pe_adj_bits,
                        int8_t *d_assign, void *stream);
int marl_envn2n_rollout(const marl_envn2n_params *p, int32_t B, int32_t T, int32_t t0, int32_t K, double *d_p_state,
                        uint8_t *d_p_active, double *d_e_state, uint8_t *d_e_active, const double *d_target,
                        int32_t *d_time_step, const int32_t *d_action_tape, const double *d_e_action_tape, uint64_t seed,
                        const marl_envn2n_records *rec, void *stream);

/* ---- kernel family 5: DHGN actor/critic, the non-GEMM parts (fp32) -----------------------------------------
 * The dense E-wide layers (AGG_vertex_0, semantic_layer, AGG_fcra_k, FCRA_layers.k, GRU weight matrices) are plain
 * library GEMMs on the host side; these entry points fuse everything pairwise / sparse / pointwise around them so that
 * no [.,N,N,8], [.,N,O,4] or dense 0/1 adjacency tensor is materialised.  E = embedding_dim in {32, 64, 128}.
 *
 * marl_dhgn_message_{fwd,bwd}: DHGN.message + L1-normalised mean aggregation of the three relations
 * (DHGN/mappo_parallel.py:256-281,323-348) from bit-packed adjacency.  S samples x N agents;
 * p f32 [S,N,4], e f32 [S,4], oxy f32 [Bo,O,2] + o_index i32 [S] + o_count i32 [Bo] (obstacle cells per map; the count
 * is what "all ones" spans for the critic: O_b during rollout, O in training — :64-65, SURVEY 7.4-5);
 * W0 [E,8], W1 [E,4], W2 [E,4] = MSG_layers.{0,1,2}.weight.  Out: agg f32 [S,N,3,E] (input of AGG_vertex_0).
 * bwd accumulates (+=) the weight/bias gradients; inputs are data, so there is no input gradient. */
int marl_dhgn_message_fwd(int32_t S, int32_t N, int32_t O, int32_t E, const float *d_p, const float *d_e,
                          const float *d_oxy, const int32_t *d_o_index, const int32_t *d_o_count,
                          const uint32_t *d_p_adj_bits, const uint8_t *d_e_adj, const uint32_t *d_o_adj_bits,
                          int32_t all_ones, const float *d_W0, const float *d_b0, const float *d_W1, const float *d_b1,
                          const float *d_W2, const float *d_b2, float *d_agg, void *stream);
int marl_dhgn_message_bwd(int32_t S, int32_t N, int32_t O, int32_t E, const float *d_p, const float *d_e,
                          const float *d_oxy, const int32_t *d_o_index, const int32_t *d_o_count,
                          const uint32_t *d_p_adj_bits, const uint8_t *d_e_adj, const uint32_t *d_o_adj_bits,
                          int32_t all_ones, const float *d_W0, const float *d_b0, const float *d_W1, const float *d_b1,
                          const float *d_W2, const float *d_b2, const float *d_grad_agg, float *d_gW0, float *d_gb0,
                          float *d_gW1, float *d_gb1, float *d_gW2, float *d_gb2, void *stream);
/* L1norm(adj) @ hist of DHGN.fcra (:204-233): out[s,i,:] = mean over neighbours j of hist[s*sample_stride + j*agent_stride]. */
int marl_fcra_agg(int32_t S, int32_t N, int32_t E, const float *d_hist, int64_t sample_stride, int64_t agent_stride,
                  const uint32_t *d_p_adj_bits, int32_t all_ones, float *d_out, void *stream);
/* torch.nn.GRU cell pointwise (gate order r,z,n) given gi = x W_ih^T + b_ih and gh = h W_hh^T + b_hh, both [R,3E]. */
int marl_gru_cell_fwd(int64_t R, int32_t E, const float *d_gi, const float *d_gh, const float *d_h_prev,
                      float *d_h_new, float *d_save_r, float *d_save_z, float *d_save_n, float *d_save_hn, void *stream);
int marl_gru_cell_bwd(int64_t R, int32_t E, const float *d_dh_new, const float *d_save_r, const float *d_save_z,
                      const float *d_save_n, const float *d_save_hn, const float *d_h_prev, float *d_dgi, float *d_dgh,
                      float *d_dh_prev, void *stream);
/* Actor softmax/Categorical + critic head + PPO-clip / clipped value losses, forward AND backward in one pass
 * (:437,446-456,526,692-706).  Adds {sum actor_term*active, sum critic_term*active, sum active} to d_sums[3] and
 * writes d(sum)/d logits [R,A], d(sum)/d value [R]; the caller divides by sum(active).  d_v_old == NULL selects the unclipped
 * value loss (values_now - v_target)^2 of use_value_clip = False (:703-704). */
int marl_ppo_head(int64_t R, int32_t E, int32_t A, const float *d_feat_a, const float *d_feat_c, const float *d_Wa,
                  const float *d_ba, const float *d_wc_eff, const float *d_bc, const float *d_action,
                  const float *d_old_logp, const float *d_adv, const float *d_v_old, const float *d_v_target,
                  const float *d_active, float eps, float ent_coef, float *d_logp, float *d_entropy, float *d_value,
                  float *d_dlogits, float *d_dvalue, float *d_sums, void *stream);
/* Rollout-time heads (:440-449, :513): softmax -> sample (counter RNG keyed by seed,row,t) or argmax -> log-prob; value. */
int marl_act_head(int64_t R, int32_t E, int32_t A, const float *d_feat_a, const float *d_feat_c, const float *d_Wa,
                  const float *d_ba, const float *d_wc_eff, const float *d_bc, uint64_t seed, int32_t t,
                  int32_t deterministic, int32_t *d_action, float *d_action_f32, float *d_logp, float *d_value,
                  void *stream);
/* Dense layer on the tcgen05 tensor cores with fp32-level accuracy (3xTF32 split, fp32 accumulation in TMEM):
 * C[M,N] = act(A1[M,K1] W[:, :K1]^T + A2[M,K2] W[:, K1:]^T + bias[N] + D[M,N]), W = nn.Linear weight [N, K1+K2] row-major.
 * Replaces the library sgemm behind every E-wide nn.Linear / GRU projection of DHGN/mappo_parallel.py:116-545.  The
 * second operand pair stands in for torch.concatenate([a, b], -1) (:232), D for the 4-wide state part of the semantic
 * layer (:286,303).  Requires N % 128 == 0, K1 % 32 == 0, K2 % 32 == 0, 16-byte aligned rows. */
int marl_gemm_tf32x3(int32_t M, int32_t N, int32_t K1, int32_t K2, const float *d_A1, int64_t lda1, const float *d_A2,
                     int64_t lda2, const float *d_W, int64_t ldw, const float *d_bias, const float *d_D, int64_t ldd,
                     float *d_C, int64_t ldc, int32_t relu, void *stream);

/* ---- fused rollout step of the DHGN actor / critic (tcgen05 + TMEM, one launch per env step) -------------------------------
 * Replaces, for all B envs at once, the network half of the rollout body DHGN/mappo_parallel.py:758-801:
 * actor.choose_action (:440-449) and critic.forward mode 0 (:510-514) — encoder (DHGN :235-348), nn.GRU step, heads.
 * All pointers are device pointers in the nn.Module layouts ([out,in] row-major).  E = embedding_dim must be 128, the GRU
 * has 2 layers, depth = algo.depth in 1..3.  For the critic, head_w is the EFFECTIVE [1,E] row (weight_orig / sigma of
 * torch.nn.utils.spectral_norm) and "all ones" adjacency is used (:64-65) over the o_count real obstacle cells. */
typedef struct marl_dhgn_weights {
    const float *msg_w[3], *msg_b[3];          /* MSG_layers.{0,1,2}: [E,8], [E,4], [E,4] */
    const float *agg_v_w, *agg_v_b;            /* AGG_layers.AGG_vertex_0 [E,E] */
    const float *sem_w, *sem_b;                /* semantic_layer [E, 3E+4] */
    const float *agg_f_w[3], *agg_f_b[3];      /* AGG_layers.AGG_fcra_k [E,E] */
    const float *fcra_w[3], *fcra_b[3];        /* FCRA_layers.k [E,2E] */
    const float *gru_w_ih[2], *gru_w_hh[2], *gru_b_ih[2], *gru_b_hh[2];   /* nn.GRU [3E,E], [3E] */
    const float *head_w, *head_b;              /* actor Mean [A,E],[A]; critic effective row [1,E],[1] */
} marl_dhgn_weights;
typedef struct marl_policy_net_io {
    const void *d_packed;        /* marl_policy_pack output (1024-byte aligned, marl_policy_pack_bytes bytes) */
    const float *d_hist[3];      /* history embeddings [B,N,E], k = 0 the most recent; NULL = zeros (:750-752) */
    float *d_emb_out;            /* [B,N,E] this step's embedding (stored at t+D of the history buffer) */
    float *d_hidden;             /* [2, B*N, E] GRU hidden state (input; also the output when d_hidden_out is NULL) */
    float *d_hidden_out;         /* NULL (update d_hidden in place) or a distinct [2, B*N, E] buffer for the new state: the caller
                                    ping-pongs the two.  Required by the two-CTA-per-SM kernel variant (its GRU runs in two
                                    column halves and re-reads the previous state) */
} marl_policy_net_io;
typedef struct marl_policy_step {
    int32_t B, N, O, E, depth, action_dim, t, deterministic;
    int32_t force_action;        /* != 0: d_action is an INPUT (teacher forcing); d_logp is the log-prob of that action */
    int32_t variant;             /* 0 = choose; 1 = one (tile, network) item per CTA (16 worker warps); 2 = two CTAs per SM; 3 = the actor and
                                    the critic chain of a tile interleaved in one CTA (both networks given); 2 and 3 need d_hidden_out */
    uint64_t seed;               /* sampling: same counter RNG as marl_act_head (keyed by seed, row, t) */
    const void *d_p_state;       /* [B,N,4] double (float with MARL_POLICY_STATE_F32) */
    const void *d_e_state;       /* [B,4] double (float with MARL_POLICY_STATE_F32) */
    const int32_t *d_oxy;        /* [M,O,2] boundary cells per map (marl_raser_map_build) */
    const int32_t *d_map_id;     /* [B] or NULL */
    const int32_t *d_o_count;    /* [M] real boundary cells per map, clamped to O */
    const uint32_t *d_p_adj_bits; const uint8_t *d_e_adj; const uint32_t *d_o_adj_bits;   /* marl_env_observe outputs */
    int32_t *d_action;           /* [B,N] out (actor) */
    float *d_logp;               /* [B,N] out (actor) */
    float *d_value;              /* [B,N] out (critic) */
    void *d_debug;               /* NULL, or i64 [grid,16] per-CTA phase cycle counters (profiling aid) */
    int64_t row_offset;          /* added to the row index in the sampling RNG key: a launch over envs [lo, hi) of a larger batch passes
                                    lo * N and draws the same actions as the whole-batch launch */
    int32_t tile_rows;           /* 0 = choose the rows per work item with the wave model (a lone launch: fill the last wave); > 0 = that
                                    many rows (a multiple of N, <= 128) - launches that run concurrently with others (env-group
                                    pipelines) use full tiles and leave SMs free for their neighbours */
    int32_t flags;               /* MARL_POLICY_* bits; any other bit set is MARL_EINVAL */
} marl_policy_step;
/* marl_policy_step.flags.  Both modes are separate kernel instantiations: flags = 0 runs exactly the default kernels.
 * STATE_F32: d_p_state / d_e_state point to float [B,N,4] / [B,4] (the rollout arena's per-step records, (float) of the fp64
 *   state - the very values the kernel converts the fp64 state to) instead of double.  Not with variant 2.
 * EMBED_ONLY: run the encoder and FCRA chain only and write d_emb_out; no GRU, cells or heads.  d_hidden, d_hidden_out,
 *   d_action, d_logp and d_value may be NULL.  Used to regenerate the history embeddings of a stored episode. */
#define MARL_POLICY_STATE_F32 1
#define MARL_POLICY_EMBED_ONLY 2
/* Pre-splits (two-term fp16: hi = fp16(w), lo = fp16(w - hi)) and pre-swizzles every dense layer of one network into the shared-memory image the fused kernel
 * streams; call once per weight update. */
int64_t marl_policy_pack_bytes(int32_t depth, int32_t is_actor);
int marl_policy_pack(const marl_dhgn_weights *w, int32_t depth, int32_t is_actor, int32_t action_dim, void *d_packed, void *stream);
/* One env step of both networks (either pair may be NULL to run only the other, e.g. the critic-only bootstrap :806-825). */
int marl_policy_rollout_step(const marl_policy_step *s, const marl_dhgn_weights *actor_w, const marl_policy_net_io *actor_io,
                             const marl_dhgn_weights *critic_w, const marl_policy_net_io *critic_io, void *stream);

/* ---- second network family: GnnExtractor (obstacle_differ_3hop/mappo_parallel.py:34-70) -------------------------------------
 * L1-normalised adjacency-weighted mean over entities (F.normalize(adj, p=1) then adj @ x, :55-66).  rows = S*N (sample, agent)
 * rows; adj f32 [rows, J] (J = N + O entities); element (s,i,j,:) of x lives at s*sample_stride + i*agent_stride +
 * j*entity_stride floats, j < jmax <= J (h0: dense [S,N,J,E] => strides (N*J*E, J*E, E), jmax = J; last_comm_embedding
 * [S,N,2E] shared by all agents of a sample => strides (N*2E, 0, 2E), jmax = N).  The weights are always normalised over all J
 * entities.  all_ones != 0: the critic's ones_like(adj) (:171).  E in {32, 64, 128, 256}.  bwd: d x for the dense h0 layout. */
int marl_entity_agg_fwd(int64_t rows, int32_t N, int32_t J, int32_t jmax, int32_t E, const float *d_adj, int32_t all_ones,
                        const float *d_x, int64_t sample_stride, int64_t agent_stride, int64_t entity_stride, float *d_out,
                        void *stream);
int marl_entity_agg_bwd(int64_t rows, int32_t J, int32_t E, const float *d_adj, int32_t all_ones, const float *d_dout, float *d_dx,
                        void *stream);

/* ---- nn.GRU layer recurrence over a whole sequence, one persistent kernel per direction (hidden size 128) ----------------------
 * Replaces the T-step loop inside torch.nn.GRU (SharedActor/SharedCritic.forward mode 1, DHGN/mappo_parallel.py:424-433,531-538)
 * and its autograd backward.  gi f32 [T,R,3E] = x W_ih^T + b_ih for all steps (one GEMM by the caller); gate order r, z, n.
 * marl_gru_pack pre-splits / pre-swizzles W_hh [3E,E] for both directions into d_packed (1024-byte aligned,
 * marl_gru_pack_bytes() bytes).  fwd: out [T,R,E] (h_t), saves [4,T,R,E] = (r, z, n, W_hn h + b_hn) for the backward (may be
 * NULL).  bwd: given d_out, writes dgi, dgh [T,R,3E] (the gradients w.r.t. gi and gh = h W_hh^T + b_hh, from which the caller
 * forms dx, dW_ih, dW_hh and the bias gradients with plain GEMMs / reductions) and dh0 [R,E]. */
int64_t marl_gru_pack_bytes(void);
int marl_gru_pack(const float *d_w_hh, void *d_packed, void *stream);
int marl_gru_seq_fwd(int32_t T, int64_t R, int32_t E, const float *d_gi, const float *d_h0, const void *d_packed,
                     const float *d_b_hh, float *d_out, float *d_saves, void *stream);
int marl_gru_seq_bwd(int32_t T, int64_t R, int32_t E, const float *d_dout, const float *d_saves, const float *d_out,
                     const float *d_h0, const void *d_packed, float *d_dgi, float *d_dgh, float *d_dh0, void *stream);

/* Weight gradient of a dense layer on the tcgen05 tensor cores (3xTF32, fp32-level accuracy, deterministic split-K):
 * dW[n][k] (+)= sum_{r<R} dY[r][n] X[r][k], dY f32 [R, N_out] (row stride lddy), X f32 [R, K_in] (row stride ldx), dW row stride
 * lddw (so the two halves of a concatenated input can be written into column ranges of one gradient); d_dbias (may be NULL)
 * f32 [N_out] receives sum_r dY[r][:] (the bias gradient) from the same loads.  Replaces the autograd
 * weight-gradient GEMMs behind `ac_loss.backward()` (DHGN/mappo_parallel.py:708).  N_out, K_in multiples of 128.
 * d_workspace: marl_wgrad_workspace_bytes(R, N_out, K_in) bytes. */
int64_t marl_wgrad_workspace_bytes(int64_t R, int32_t N_out, int32_t K_in);
int marl_wgrad_tf32x3(int64_t R, int32_t N_out, int32_t K_in, const float *d_dY, int64_t lddy, const float *d_X, int64_t ldx,
                      float *d_dW, int64_t lddw, float *d_dbias, int32_t accumulate, void *d_workspace, void *stream);

/* Persistent row-tile GEMM for training (forward and input-gradient GEMMs of every E-wide layer), tcgen05 3xTF32:
 * C[M,N] = act([A1 | A2] B^T + bias + D), B[N, K1+K2] given pre-packed by marl_rowgemm_pack from any strided view
 * (B[n][k] = d_W[n*stride_n + k*stride_k]: an nn.Linear weight as is, or its transpose for dX = dY W).  N <= 512 and all of
 * N, K1, K2 multiples of 128 (K2 may be 0); rows 16-byte aligned.  d_packed: 1024-byte aligned, marl_rowgemm_pack_bytes(N, K). */
int64_t marl_rowgemm_pack_bytes(int32_t N, int32_t K);
int marl_rowgemm_pack(const float *d_W, int64_t stride_n, int64_t stride_k, int32_t N, int32_t K, void *d_packed, void *stream);
int marl_rowgemm_tf32x3(int64_t M, int32_t N, int32_t K1, int32_t K2, const float *d_A1, int64_t lda1, const float *d_A2, int64_t lda2,
                        const void *d_packed, const float *d_bias, const float *d_D, int64_t ldd, float *d_C, int64_t ldc, int32_t relu,
                        void *stream);

/* Training-side helpers behind `ac_loss.backward()` (DHGN/mappo_parallel.py:708).
 * marl_relu_bwd: d_dst = d_out > 0 ? d_dy : 0 over n floats (backward of a ReLU fused into a GEMM epilogue; n % 4 == 0, 16-byte aligned).
 * marl_skinny_wgrad: weight (and bias) gradient of a layer whose input is K_in <= 16 wide - the state part of the semantic layer
 * (:286,303), or, with the roles of the operands swapped, the 9-row actor head (:437): dW[n][k] = sum_r dY[r][n] P[r][k] written with row stride lddw (e.g. straight into columns 0..3 of the [E, 3E+4]
 * gradient), d_dbias[n] = sum_r dY[r][n] (may be NULL).  Deterministic (fixed row slices, ordered reduction).
 * d_workspace: marl_skinny_wgrad_workspace_bytes(R, N_out, K_in) bytes. */
int marl_relu_bwd(int64_t n, const float *d_dy, const float *d_out, float *d_dst, void *stream);
int64_t marl_skinny_wgrad_workspace_bytes(int64_t R, int32_t N_out, int32_t K_in);
int marl_skinny_wgrad(int64_t R, int32_t N_out, int32_t K_in, const float *d_dY, int64_t lddy, const float *d_P, int64_t ldp,
                      float *d_dW, int64_t lddw, float *d_dbias, void *d_workspace, void *stream);

/* torch.nn.utils.clip_grad_norm_ (:710-711) and torch.optim.Adam.step (runner.py:72-78) on flat fp32 arenas. */
int64_t marl_clip_workspace_bytes(int64_t n);
int marl_clip_grad_norm(int64_t n, float *d_grad, float max_norm, void *d_workspace, float *d_total_norm, void *stream);
int marl_adam_step(int64_t n, float *d_param, const float *d_grad, float *d_exp_avg, float *d_exp_avg_sq, float lr,
                   float beta1, float beta2, float eps, int64_t step, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MARL_B200_H */

/*
 * cbev.h -- C ABI of the B200-native CarlaBEV batched stepping engine.
 *
 * The reference (danielmtzbarba/carlabev-env) has no FFI: its boundary for this path is the
 * gymnasium VectorEnv returned by CarlaBEV.envs.make_env (envs/__init__.py:108-120), i.e.
 * SyncVectorEnv.reset / SyncVectorEnv.step over CarlaBEV.reset / CarlaBEV.step
 * (envs/carlabev.py:96-148, 223-231) plus the wrap_env chain (envs/__init__.py:40-90).
 * The entry points below are what a binding behind that Python surface calls; each cites the
 * reference interface it replaces.  Plain pointers and sizes only -- no torch types.
 *
 * Ownership: the engine owns its opaque handle, the uploaded map / scene pool and the per-env
 * struct-of-arrays state.  The caller owns every I/O buffer (actions, observation ring, rewards,
 * flags, info blocks) and the CUDA stream.  All calls are asynchronous on `stream` unless stated.
 * Every function returns 0 on success or a CBEV_ERR_* code; cbev_last_error() gives the message
 * (thread-local).  One host thread per engine.
 */
#ifndef CBEV_H
#define CBEV_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CBEV_VERSION 201

/* ---- error codes -------------------------------------------------------------------------- */
#define CBEV_OK 0
#define CBEV_ERR_ARG 1      /* invalid argument / configuration (ValueError in the reference) */
#define CBEV_ERR_CUDA 2     /* CUDA runtime failure                                           */
#define CBEV_ERR_STATE 3    /* call order violated (e.g. step before reset, no pool)          */
#define CBEV_ERR_NOMEM 4

/* ---- enums -------------------------------------------------------------------------------- */
/* observation modes: EnvConfig.obs_mode + wrap_env (config/env.py:27, envs/__init__.py:62-83) */
#define CBEV_OBS_SEMANTIC 0  /* float32 (F*C, oh, ow): Resize -> SemanticMask -> FrameStack -> Flatten */
#define CBEV_OBS_GRAY 1      /* uint8   (F, oh, ow):   Resize -> Grayscale -> FrameStack               */
#define CBEV_OBS_RGB 2       /* uint8   (S, S, 3):     raw CarlaBEV.render() frame (spaces.py:56-59)    */
#define CBEV_OBS_SEMANTIC_U8 3 /* uint8 (F*C, oh, ow): the masks of CBEV_OBS_SEMANTIC as 0 / 1 bytes
                                  (an extension beyond the reference: 1/4 of the ring and of the store traffic) */

/* semantic_mask_ch (wrappers/rgb_to_semantic.py:6-42) */
#define CBEV_MASK_BINARY 0
#define CBEV_MASK_2 1
#define CBEV_MASK_4 2
#define CBEV_MASK_5 3
#define CBEV_MASK_6 4
#define CBEV_MASK_7 5

#define CBEV_ACTION_DISCRETE 0   /* int64 ids into discrete_table (config/action_profiles.py:35-76) */
#define CBEV_ACTION_CONTINUOUS 1 /* float32[3] gas, steer, brake (envs/spaces.py:27-47)             */

#define CBEV_REWARD_CARL 0     /* src/deeprl/carl_reward_fn.py */
#define CBEV_REWARD_SHAPING 1  /* src/deeprl/reward.py         */

#define CBEV_AUTORESET_DISABLED 0  /* reference behaviour: caller resets with a mask              */
#define CBEV_AUTORESET_NEXT_STEP 1 /* device auto-reset from the pool on the step after a terminal */

/* palette indices used by frames, draw lists and traffic lights (semantics.py:19-28) */
#define CBEV_PAL_NON_DRIVABLE 0
#define CBEV_PAL_DRIVABLE 1
#define CBEV_PAL_SIDEWALK 2
#define CBEV_PAL_VEHICLE 3
#define CBEV_PAL_PEDESTRIAN 4
#define CBEV_PAL_ROUTE 5
#define CBEV_PAL_TL_RED 6
#define CBEV_PAL_TL_YELLOW 7
#define CBEV_PAL_BLACK 8
#define CBEV_PAL_TL_OFF 9
#define CBEV_PAL_COUNT 10

/* termination causes (envs/carlabev.py:43-49 plus the non-terminal "ckpt") */
#define CBEV_CAUSE_NONE 0
#define CBEV_CAUSE_CKPT 1
#define CBEV_CAUSE_COLLISION 2
#define CBEV_CAUSE_SUCCESS 3
#define CBEV_CAUSE_OUT_OF_BOUNDS 4
#define CBEV_CAUSE_OFF_ROAD 5
#define CBEV_CAUSE_MAX_ACTIONS 6
#define CBEV_CAUSE_COUNT 8

/* behaviours of scripted actors (src/actors/behavior/) */
#define CBEV_BEH_NONE 0
#define CBEV_BEH_LEAD_BRAKE 1
#define CBEV_BEH_CROSS 2
#define CBEV_BEH_STOP_MID 3
#define CBEV_BEH_STOP_RETURN 4

/* ---- per-step "hero" info block: info["hero"] / info["collision"] of the reference
 *      (stanley_controller.py:163-176, hero.py:119-138, scene.py:207-225), CBEV_HERO_FIELDS doubles/env */
enum {
  CBEV_H_X = 0, CBEV_H_Y, CBEV_H_YAW, CBEV_H_V,                 /* state            */
  CBEV_H_X1, CBEV_H_Y1, CBEV_H_YAW1, CBEV_H_V1,                 /* last_state       */
  CBEV_H_DIST2WP, CBEV_H_SP_X, CBEV_H_SP_Y, CBEV_H_SP_YAW,      /* dist2wp, set_point */
  CBEV_H_CMD_GAS, CBEV_H_CMD_STEER, CBEV_H_CMD_BRAKE, CBEV_H_DELTA,
  CBEV_H_SPEED_MPS, CBEV_H_ACCEL_LONG, CBEV_H_ACCEL_LAT, CBEV_H_JERK_LONG, CBEV_H_JERK_LAT,
  CBEV_H_YAW_RATE, CBEV_H_YAW_ACC,
  CBEV_H_ACC, CBEV_H_TIDX, CBEV_H_HIT, CBEV_H_HIT_ID, CBEV_H_TILE, CBEV_H_NEARBY,
  CBEV_H_DIST2GOAL, CBEV_H_T, CBEV_H_SCENE,
  CBEV_HERO_FIELDS
};

/* ---- episode summary written on terminal steps (stats.py:127-148, carlabev.py:177-185) */
enum {
  CBEV_E_RETURN = 0, CBEV_E_LENGTH, CBEV_E_CAUSE, CBEV_E_MEAN_SPEED,
  CBEV_E_ABS_ACCEL_LONG, CBEV_E_ABS_ACCEL_LAT, CBEV_E_ABS_JERK_LONG, CBEV_E_ABS_JERK_LAT,
  CBEV_E_ABS_YAW_RATE, CBEV_E_ABS_YAW_ACC, CBEV_E_VIOL_RATE, CBEV_E_HARSH_RATE,
  CBEV_E_SCENE, CBEV_E_NUM_VEHICLES, CBEV_E_LEN_ROUTE, CBEV_E_EPISODE,
  CBEV_EPISODE_FIELDS
};

/* ---- global episode statistics (the only cross-GPU reduction; stats.py:19-148) */
enum {
  CBEV_S_EPISODES = 0, CBEV_S_RETURN, CBEV_S_LENGTH, CBEV_S_MEAN_SPEED,
  CBEV_S_CAUSE0, /* CBEV_CAUSE_COUNT counters */
  CBEV_S_ABS_COMFORT0 = CBEV_S_CAUSE0 + CBEV_CAUSE_COUNT, /* 6 sums of per-episode mean |metric| */
  CBEV_S_VIOL_RATE = CBEV_S_ABS_COMFORT0 + 6, CBEV_S_HARSH_RATE, CBEV_S_STEPS,
  CBEV_STATS_FIELDS
};

/* ---- configuration ------------------------------------------------------------------------ */
typedef struct {
  int32_t num_envs;
  int32_t fov_size;          /* EnvConfig.size, 128                                  */
  double anchor_x_frac;      /* EnvConfig.ego_anchor_x_frac (fov.py:30-36)           */
  double anchor_y_frac;
  int32_t obs_h, obs_w;      /* EnvConfig.obs_size: (96, 96) default; any 8..128 per side (cv2 INTER_AREA), h*w % 4 == 0 (float masks) / % 16 == 0 (gray, uint8 masks) */
  int32_t obs_mode;          /* CBEV_OBS_*                                           */
  int32_t mask_mode;         /* CBEV_MASK_*                                          */
  int32_t frame_stack;       /* EnvConfig.frame_stack                                */
  int32_t ring_slots;        /* L >= frame_stack + 1 slots per env in the obs ring   */
  int32_t action_mode;       /* CBEV_ACTION_*                                        */
  int32_t n_discrete;        /* rows of discrete_table                               */
  float discrete_table[16 * 3];
  int32_t reward_mode;       /* CBEV_REWARD_*                                        */
  int32_t autoreset;         /* CBEV_AUTORESET_*                                     */
  int32_t max_actors;        /* capacity of the per-env actor arrays (>= pool max)   */
  int32_t trajectory_steps;  /* steps of open-loop actor trajectory rolled out per scene at pool upload (0 = off) */
  /* CaRL parameters (carl_reward_fn.py:73-88; config/reward_profiles.py) */
  double lane_center_exponent, lane_center_floor, off_lane_penalty;
  double speed_penalty_scale, speed_penalty_floor, ttc_threshold, ttc_penalty_floor;
  /* shaping parameters (reward.py:14-47) */
  int32_t max_actions, offroad_terminate_after;
  double sidewalk_step_penalty, sidewalk_penalty_scale;
  double k_lat_quadratic, k_progress, k_flow, k_align_bonus, k_reverse, k_ttc, alive_bias;
  double k_smooth, k_steer_smooth, k_steer_jerk, k_route_dev, route_dev_start;
  double max_speed_for_flow, lat_clip, yaw_small, lat_small;
  uint64_t seed;             /* seeds the device auto-reset scene draw               */
} cbev_config;

/* Scene pool, flat host arrays (carlabev_env_b200/pool.py:pack_pool; SURVEY.md Appendix B).
 * Replaces SceneGenerator.build_scene + Scene.load_scene at reset (scene_generator.py:95,
 * scenes/scene.py:61-88): scenes are pre-generated on the host and made device resident. */
typedef struct {
  int32_t n_scenes;
  int32_t n_actors_total, n_tl_total;
  /* per scene */
  const double* ego_state0;       /* [n][4] x, y, yaw, v (post-reset)          */
  const double* ego_target_speed; /* [n] px/s                                   */
  const int32_t* ego_tidx0;       /* [n]                                        */
  const double* len_ego_route;    /* [n]                                        */
  const int32_t* num_vehicles;    /* [n]                                        */
  const int32_t* ego_off;         /* [n+1] into ego_cx/cy/cyaw                  */
  const int32_t* rew_off;         /* [n+1] into rew_rx/ry/cum                   */
  const int32_t* actor_off;       /* [n+1] into per-actor arrays                */
  const int32_t* tl_off;          /* [n+1] into tl_rect/tl_color                */
  /* routes */
  const double *ego_cx, *ego_cy, *ego_cyaw;
  const int32_t *rew_rx, *rew_ry;
  const double* rew_cum;          /* cumulative lengths (carl_reward_fn.py:20-26) */
  /* per actor */
  const uint8_t* act_kind;        /* 0 vehicle, 1 pedestrian                     */
  const double* act_state0;       /* [.][4]                                      */
  const int32_t* act_tidx0;
  const double *act_cruise_px, *act_cruise_mps;
  const uint8_t* act_beh;         /* CBEV_BEH_*                                  */
  const double* act_beh_p;        /* [.][4]                                      */
  const int32_t* act_route_off;   /* [n_actors_total+1]                          */
  const int32_t* act_raw_off;     /* [n_actors_total+1]                          */
  const double *act_cx, *act_cy, *act_cyaw;
  const double *act_raw_x, *act_raw_y;
  /* traffic lights */
  const int32_t* tl_rect;         /* [.][4] x, y, w, h as drawn (unpadded coords) */
  const uint8_t* tl_color;        /* CBEV_PAL_*                                   */
  /* small-route Savitzky-Golay matrices for the mid-episode retreat (jaywalk.py:43-54):
   * sg_mat[n] is the n x n linear operator of savgol_filter for an n-point route, n <= CBEV_SG_MAX */
  const double* sg_mat;           /* [CBEV_SG_MAX+1][CBEV_SG_MAX][CBEV_SG_MAX], may be NULL */
} cbev_pool_desc;
#define CBEV_SG_MAX 12

/* Device output pointers of one step (all nullable except reward/terminated/truncated). */
typedef struct {
  double* reward;       /* [N]  SyncVectorEnv rewards are float64                    */
  uint8_t* terminated;  /* [N]                                                       */
  uint8_t* truncated;   /* [N]                                                       */
  uint8_t* cause;       /* [N]  CBEV_CAUSE_*                                         */
  double* hero;         /* [N][CBEV_HERO_FIELDS]                                     */
  double* episode;      /* [N][CBEV_EPISODE_FIELDS], rows written on terminal steps  */
} cbev_step_out;

typedef struct cbev_engine* cbev_handle;

/* lifecycle -- replaces make_env / CarlaBEV.__init__ (envs/__init__.py:108-120, carlabev.py:51-72) */
int cbev_version(void);
const char* cbev_last_error(void);
int cbev_create(const cbev_config* cfg, cbev_handle* out);
int cbev_destroy(cbev_handle h);

/* BaseMap.__init__ / load_map (envs/world.py:33-67, envs/utils.py:49-62): class map, 1 byte/pixel
 * (0 non-drivable, 1 drivable, 2 sidewalk), row pitch = w.  Synchronous. */
int cbev_upload_map(cbev_handle h, const uint8_t* cls_host, int32_t w, int32_t h_px);

/* SceneGenerator output made device resident (see cbev_pool_desc).  Synchronous. */
int cbev_upload_scene_pool(cbev_handle h, const cbev_pool_desc* pool);

/* Row f2: the scripted scenarios generated ON THE DEVICE from (kind, level, scene_seed) -- SceneGenerator.build_scene
 * for scene in {"lead_brake", "jaywalk"} (scene_generator.py:171-182 -> scenarios/lead_brake.py:18-129,
 * scenarios/jaywalk.py:29-117) followed by Scene.load_scene with its spawn jitter and CarlaBEV.reset's validation /
 * retry loop (carlabev.py:108-131).  One thread per scene: sha256-derived sub-seeds (randomness.py:13-16),
 * np.random.default_rng = SeedSequence -> PCG64, Generator.integers / uniform in the reference's draw order.  The
 * result replaces the engine's pool exactly like cbev_upload_scene_pool (append-only while envs are running).
 * kinds[i]: 1 lead_brake (levels 1-3), 2 jaywalk (levels 1-4); sg_mat as in cbev_pool_desc; attempts_host (nullable)
 * receives the number of samples each scene needed.  Drawn parameters, raw routes, behaviour parameters and spawn
 * jitter are bit-identical to the reference; smoothed routes agree to ~1e-12 px (SciPy's LAPACK edge fit is not
 * reproducible operation for operation).  Synchronous. */
int cbev_generate_scenes(cbev_handle h, int32_t n, const uint8_t* kinds, const int32_t* levels, const int64_t* seeds,
                         const double* sg_mat, int32_t* attempts_host);

/* Debug / parity: sizes of the resident pool -- n_scenes, n_actors, ego route points, reward route points, actor
 * route points, authored route points, traffic lights, rolled-out trajectory steps -- and a read-back of its arrays
 * into the HOST buffers of a cbev_pool_desc (NULL members are skipped; sg_mat is not read back). */
int cbev_pool_counts(cbev_handle h, int32_t counts[8]);
int cbev_read_scene_pool(cbev_handle h, const cbev_pool_desc* dst_host);

/* Observation ring owned by the caller: ring_slots frames per env, env-major.
 * frame bytes = cbev_frame_bytes(); layout [N][ring_slots][frame]. */
int64_t cbev_frame_bytes(cbev_handle h);
int cbev_bind_obs_ring(cbev_handle h, void* ring_dev, int64_t bytes);

/* SyncVectorEnv.reset(options={"reset_mask": m}) -> CarlaBEV.reset (gymnasium vector reset;
 * carlabev.py:96-148).  mask_dev: uint8[N] or NULL (= all); scene_ids_dev: int32[N] pool indices
 * (read where mask is set).  Renders the actor-less reset frame (world.py:92-100) into all
 * frame_stack window slots (FrameStackObservation padding_type="reset"). */
int cbev_reset(cbev_handle h, const uint8_t* mask_dev, const int32_t* scene_ids_dev, void* stream);

/* SyncVectorEnv.step(actions) -> CarlaBEV.step (carlabev.py:223-231) for all envs.
 * actions_dev: int64[N] (discrete) or float32[N][3] (continuous).  Advances the ring head. */
int cbev_step(cbev_handle h, const void* actions_dev, const cbev_step_out* out, void* stream);

/* Same, with HOST (pinned) buffers: copies actions H2D, steps, copies reward / terminated /
 * truncated back D2H on `stream`; the observation stays device resident.  If the three outputs are laid
 * out back to back (terminated_host == reward_host + 8N bytes, truncated_host == terminated_host + N) they
 * come back in a single copy. */
int cbev_step_host(cbev_handle h, const void* actions_host, double* reward_host, uint8_t* terminated_host,
                   uint8_t* truncated_host, void* stream);

/* Host (pinned) destinations of one step.  reward / terminated / truncated are required; episode (the
 * [N][CBEV_EPISODE_FIELDS] block, rows of finished envs are valid) and cause are optional.  If reward, terminated
 * and truncated are laid out back to back they come back in one copy. */
typedef struct {
  double* reward;
  uint8_t* terminated;
  uint8_t* truncated;
  uint8_t* cause;
  double* episode;
} cbev_host_out;

/* cbev_step_host with caller-owned DEVICE outputs as well (dev_out may be NULL: internal staging, reward and flags
 * only) and the optional host copies of cbev_host_out.  The D2H copies are issued on a side stream as soon as the
 * simulation kernels of the step have finished, i.e. they overlap the raster kernel; `stream` is made to wait for
 * them, and cbev_wait_host_outputs() blocks the calling thread until they have landed (without waiting for the
 * raster kernel) -- what SyncVectorEnv.step's caller needs before it can look at rewards / dones
 * (gymnasium vector step; envs/__init__.py:116-119). */
int cbev_step_host_ex(cbev_handle h, const void* actions_host, const cbev_step_out* dev_out,
                      const cbev_host_out* host, void* stream);
/* cbev_step with DEVICE actions (a policy on the GPU) plus the host copies a cbev_host_out describes; host may be NULL. */
int cbev_step_ex(cbev_handle h, const void* actions_dev, const cbev_step_out* dev_out, const cbev_host_out* host,
                 void* stream);
/* Action repeat (frame skip): every later cbev_step, cbev_step_ex, cbev_step_host and cbev_step_host_ex call is one
 * agent step of up to `repeat` simulator steps with the same action, and renders one frame.  For each env:
 *   - an env whose last agent step was terminal under CBEV_AUTORESET_NEXT_STEP auto-resets as before (reward 0,
 *     flags 0, the reset frame in every window slot, the reset's hero block; no simulator step runs);
 *   - every other env takes sub-steps 1..j, j the first sub-step that is terminated or truncated, or `repeat`.  Each
 *     sub-step is bit-identical to one step at repeat 1.  reward = r1 + r2 + ... + rj in double, added in sub-step
 *     order from r1 and unfused (j = 1 returns r1 bit for bit); terminated, truncated, cause, the hero block, the
 *     episode block and the statistics vector are those of sub-step j, so episode lengths count simulator steps.
 *     The one new frame is the one repeat 1 shows after sub-step j, and the window holds the last F agent-step frames.
 * The step counter (CBEV_S_STEPS) counts calls.  repeat must lie in [1, CBEV_MAX_ACTION_REPEAT] (the cap bounds how
 * long one launch runs); the default 1 keeps the three-launch step.  A repeat above 1 issues two launches per step,
 * the fused k_step_repeat and the raster kernel, and cbev_profile_read_ex reports k_step_repeat as move_ms and 0 as
 * judge_ms.  It takes effect at the next step call and has no effect on cbev_reset, snapshot / restore or the
 * lookahead calls (one simulator step per action row). */
#define CBEV_MAX_ACTION_REPEAT 64
int cbev_set_action_repeat(cbev_handle h, int32_t repeat);
/* After replacing the pool with an unrelated one: every env must be reset (with mask = NULL) before the next step. */
int cbev_invalidate(cbev_handle h);
int cbev_wait_host_outputs(cbev_handle h);

/* fov_masked (envs/fov.py:46-68, 96-99): static corner mask blitted over the composed frame before the ego
 * square is drawn.  mask_host: uint8[S*S], non-zero = pixel is painted black; NULL removes the mask.  Synchronous. */
int cbev_upload_fov_mask(cbev_handle h, const uint8_t* mask_host);

/* Temporal fusion of the stacked semantic observation (wrappers/rgb_to_semantic.py:152-193, 275-332):
 *   CBEV_FUSE_VEHICLE_TEMPORAL: current channels without the vehicle channel + vehicle_t, vehicle_t-1, vehicle_t-2
 *                               -> [N][C-1+3][oh][ow] in the ring's element type: float32 (CBEV_OBS_SEMANTIC) or
 *                                  uint8 0 / 1 (CBEV_OBS_SEMANTIC_U8)
 *   CBEV_FUSE_VEHICLE_WEIGHTED: current channels without vehicle + clip(1.0 v_t + 0.5 v_t-1 + 0.25 v_t-2, 0, 1)
 *                               -> float32 [N][C][oh][ow] for both modes (the values are not 0 / 1), bit-identical
 * Reads the current window of the ring, writes the caller-owned `out_dev`. */
#define CBEV_FUSE_VEHICLE_TEMPORAL 1
#define CBEV_FUSE_VEHICLE_WEIGHTED 2
int cbev_fuse(cbev_handle h, int32_t mode, void* out_dev, void* stream);

/* Ring head: observation of env e = slots [head - frame_stack + 1, head] of its ring row. */
int cbev_obs_head(cbev_handle h, int32_t* head);

/* Debug / parity access to the SoA state (host buffers, synchronous).
 * ego: [N][16] doubles  x,y,yaw,v,x1,y1,yaw1,v1,acc,tidx,t,dist2goal,dist2goal_1,s_prev,tgt_lo,tgt_hi
 * actors: [N][max_actors][8] doubles  x,y,yaw,v,tidx,fsm,target_mps,alive */
int cbev_get_state(cbev_handle h, double* ego_host, double* actors_host);
int cbev_set_ego_state(cbev_handle h, const double* ego_host);
/* Both blocks in the layout of cbev_get_state (either may be NULL).  Actor columns written: x, y, yaw, v, tidx, fsm,
 * target_mps and the raw flags byte (column 7).  Actors are stepped from this state only while they run live
 * (trajectory_steps = 0, or past the rolled-out steps): table look-ups are functions of (scene, step). */
int cbev_set_state(cbev_handle h, const double* ego_host, const double* actors_host);

/* Snapshot / restore of whole environments (ALE cloneState / restoreState): device-side, asynchronous on `stream`.
 * A snapshot row holds everything that decides an env's future outputs -- scene, episode counter, done flag, the ego,
 * target-visibility and episode-accumulator state, every actor array, the retreat routes, and the F frames of the
 * env's current observation window (oldest first); layout in csrc/engine.h.  Not in a row: the engine-wide statistics
 * vector and step counter, the last step's outputs, the kept palette frame, and the (result-neutral) k_move order.
 *
 * Restoring row r into env e makes e continue exactly as the env the row was taken from did, given the same actions
 * -- including trajectory-table hand-over, retreat routes and ring wraps.  Restoring into a DIFFERENT env (cloning)
 * is allowed: the clone follows its source until its next device auto-reset, whose scene draw hashes (seed, env,
 * episode) and therefore differs from the source's.  The window frames are written in place into the current
 * window slots of the ring (and their mirror slots), so zero-copy views of those envs' observations change.
 *
 * Rows belong to the engine that took them and to its pool epoch: an append-only pool extension keeps them valid
 * (a row taken with fewer retreat slots restores with the extra slots zeroed); cbev_invalidate or a non-extending
 * pool upload ends the epoch, and restore then fails with CBEV_ERR_STATE.  Both calls fail with CBEV_ERR_STATE before
 * the first reset.  Issue them on the stream the engine steps on.  Host arguments are validated before any launch;
 * device index arrays are trusted (the kernels skip env >= N and row >= n_rows). */
typedef struct {
  uint64_t engine_token;  /* random per cbev_create: rows restore only into the engine that took them */
  int32_t pool_epoch;     /* bumped by cbev_invalidate / a non-extending pool upload                  */
  int32_t retreat_slots;  /* R when the rows were taken                                                */
  int64_t row_bytes;      /* bytes per row (16-byte multiple)                                          */
  int32_t n_rows, reserved;
} cbev_snapshot_info;
/* Bytes of one snapshot row at the current number of retreat slots per env. */
int64_t cbev_snapshot_row_bytes(cbev_handle h);
/* Row i of dst_dev (16-byte aligned, >= n * row_bytes) <- env env_ids_dev[i] (NULL: env i), n in 1..N. */
int cbev_snapshot(cbev_handle h, const int32_t* env_ids_dev, int32_t n, void* dst_dev, int64_t dst_bytes,
                  cbev_snapshot_info* info_out, void* stream);
/* Env env_ids_dev[i] (NULL: env i) <- row rows_dev[i] (NULL: row i, then n <= info->n_rows) of src_dev, n in 1..N.
 * Several targets may share one row (cloning); two entries must not name the same env. */
int cbev_restore(cbev_handle h, const cbev_snapshot_info* info, const void* src_dev, const int32_t* rows_dev,
                 const int32_t* env_ids_dev, int32_t n, void* stream);

/* Observation-free lookahead (planning with the simulator as the model: MPC, CEM, MCTS rollouts).  B branches, each
 * starting from the CURRENT state of a live env, take H steps of actions without rendering, and return their rewards;
 * the live engine is left as it was.
 *
 * Same arithmetic as stepping: a branch step runs the code of cbev_step minus rendering -- action decode and
 * clipping, ego physics, scripted actors (trajectory tables, the hand-over to live stepping at trajectory_steps, live
 * behaviour FSMs and retreat routes), collisions, target consumption, CaRL or shaping reward and termination
 * (including shaping's max_actions truncation).  reward[t], the flags, the cause and the hero block of a branch are
 * therefore bit-identical to what stepping that env with the same actions would produce.
 *
 * No side effects on the live engine: the call never writes the env state, the observation ring, the render
 * descriptors or env orders, the statistics vector (cbev_read_stats), the last step's output buffers, the ring head or
 * the step counter.  A branch never auto-resets and never renders.  cbev_launch_count grows by the launches issued.
 *
 * Roots may repeat (one env cloned into many branches).  A root whose last step was terminal (it waits for a reset)
 * gives a branch with steps = 0 and ret = 0.  Fails with CBEV_ERR_STATE before the first reset (or after
 * cbev_invalidate).  Host arguments are validated before any launch; the device root array is trusted: a root outside
 * [0, N) gives steps = 0 and nothing is written out of bounds.
 *
 * Issued on `stream`, which must be the stream the engine steps on: the call is ordered after the previous step (whose
 * side-stream work that stream has already joined).  The branch state is engine-owned device memory, allocated on first
 * use, grown synchronously when B or the pool's retreat-slot count grows, and freed by cbev_destroy. */
typedef struct {
  double* ret;          /* [B] required: sum over t < steps of w_t * r_t, w_0 = 1, w_{t+1} = w_t * gamma, in step order */
  double* reward;       /* [H][B] nullable: reward of step t; exactly 0.0 for t >= steps                             */
  int32_t* steps;       /* [B] nullable: steps taken, 1..H (0 when the root's last step was terminal)               */
  uint8_t* terminated;  /* [B] nullable: flags and cause of the branch's last step taken (0 when steps == 0)        */
  uint8_t* truncated;
  uint8_t* cause;       /* CBEV_CAUSE_*                                                                            */
  double* hero;         /* [B][CBEV_HERO_FIELDS] nullable: hero block after the branch's last step taken (zeros when
                           steps == 0)                                                                             */
} cbev_lookahead_out;

/* Branch b starts from the current state of env root_env_ids_dev[b] (NULL: env b, then B <= N) and takes actions
 * actions_dev[t][b] (int64 [H][B] discrete, float32 [H][B][3] continuous) for t = 0..H-1, stopping after its first
 * terminated or truncated step.  No observation, no auto-reset; live envs, ring, statistics untouched. */
int cbev_lookahead(cbev_handle h, const int32_t* root_env_ids_dev, int32_t n_branches, int32_t horizon,
                   const void* actions_dev, double gamma, const cbev_lookahead_out* out, void* stream);

/* cbev_lookahead plus the observation window at each branch's leaf (planners that value the leaf state from its
 * observation: a learned terminal value V(obs_H), bootstrapped returns, a policy prior at the end of each rollout).
 * Same arguments and the same results in `out` -- ret, reward, steps, flags, cause and hero are bit-identical to
 * cbev_lookahead -- and in obs_dev ([B][F][cbev_frame_bytes], F = frame_stack, 1 for CBEV_OBS_RGB) the leaf window
 * of branch b, oldest frame first, byte-identical to the observation window of an env cloned from the root and stepped
 * with the branch's actions for s = steps[b] steps (auto-reset disabled):
 *   position f >= F - min(s, F): the branch's own frame of step s - F + f (0-based), rendered by the raster kernel of
 *                                the live step from the branch state after that step (a branch that ends at s < H
 *                                shows its terminal frame, as stepping does before any reset);
 *   position f <  F - s:         frame f + s of the root's current window, copied from the ring as it is (reset
 *                                frames and mirror-zone frames included).
 * s = 0 with a terminal root gives the root's current window; s = 0 with a device root outside [0, N) gives a window
 * of zero bytes (nothing is read or written out of bounds).
 *
 * No side effects, as for cbev_lookahead: the live env state, the ring, the render descriptors and draw lists, the env
 * orders and their counters, the statistics, the ring head, the step counter, the kept palette frame and the trace
 * buffer are not written.  The branches' draw records live in engine-owned device memory (staging and render
 * positions, about 2 * F * (80 + 8 * max_rects) bytes per branch), allocated on first use, grown synchronously when B
 * or max_rects (a pool upload with more traffic lights) grows, and freed by cbev_destroy.
 *
 * Host checks before any launch, each error naming its rule: those of cbev_lookahead; out->steps non-null (the window
 * copy reads it on the device); obs_dev non-null and 16-byte aligned; obs_bytes >= B * F * cbev_frame_bytes; an
 * observation ring bound.  CBEV_ERR_STATE before the first reset.  Issued on `stream` (the engine's step stream) as
 * three launches -- the branches with their draw records, the raster kernel over the B * F leaf positions, the copy
 * of the root frames -- so cbev_launch_count grows by 3. */
int cbev_lookahead_obs(cbev_handle h, const int32_t* root_env_ids_dev, int32_t n_branches, int32_t horizon,
                       const void* actions_dev, double gamma, const cbev_lookahead_out* out, void* obs_dev,
                       int64_t obs_bytes, void* stream);

/* The general lookahead (tree search, beam search, iterative deepening): branches may start from snapshot rows
 * instead of live envs, and each branch's leaf may come back as a snapshot row, which restores into a live env
 * (cbev_restore) or serves as the root of the next call.  Either way the leaf continues bit-identically.
 *
 * Roots from rows (src_info non-NULL): branch b starts from row roots[b] (NULL: row b, then B <= src_info->n_rows) of
 * src_rows.  Every output -- ret, reward, steps, flags, cause, hero and the leaf window -- is bit-identical to restoring
 * that row into an env and calling cbev_lookahead / cbev_lookahead_obs from it: the frames older than the branch's
 * first step come from the row's frame section.  A row with done = 1 gives steps = 0 and its own frames as the leaf
 * window; a device root outside [0, n_rows), or a row whose header scene lies outside the pool, gives steps = 0 and a
 * zero window (no row content makes the kernels read outside the pool).  The rows follow cbev_restore's rules: they
 * must come from this engine and its current pool epoch (CBEV_ERR_STATE otherwise), and rows taken at fewer retreat
 * slots are read with the extra slots zeroed.  src_rows is only read, and may be the same memory as leaf_rows.
 *
 * Leaf rows (leaf_rows non-NULL): row b of leaf_rows gets branch b's leaf as a full snapshot row in the engine's
 * current layout (header, the 16 state sections, the F window frames), byte-identical, padding included, to
 * cbev_snapshot of an env cloned from the root, stepped with the branch's actions for steps[b] steps (auto-reset
 * disabled) and snapshotted right after its last step: a terminal leaf has done = 1, episode + 1 and zeroed episode
 * accumulators, a non-terminal one carries them.  A steps = 0 branch from a valid root gives exactly the root's row; a
 * branch whose device root is invalid leaves its row unwritten.  *leaf_info gets the engine token, the current pool
 * epoch and retreat slots, row_bytes and n_rows = B.  Leaf rows always carry their frames, so asking for them renders
 * the leaf windows (into engine-owned scratch of B * F * cbev_frame_bytes when obs is NULL, grown synchronously and
 * freed by cbev_destroy).  A row costs cbev_snapshot_row_bytes: about 885 KB with float32 6-class masks at 96 x 96 and
 * F = 4, 222 KB with uint8 masks.
 *
 * With src_info NULL and leaf_rows NULL the call is cbev_lookahead (obs NULL) or cbev_lookahead_obs.  No side effects,
 * as for those: nothing of the live engine is written and nothing synchronises (except the first-use or growth of the
 * engine-owned buffers).  Host checks before any launch, each error naming its rule: those of cbev_lookahead; io
 * non-NULL; src_rows non-NULL and 16-byte aligned with src_info, whose retreat slots and row_bytes must match the
 * engine's layout; obs 16-byte aligned with obs_bytes >= B * F * cbev_frame_bytes; leaf_rows 16-byte aligned with
 * leaf_bytes >= B * cbev_snapshot_row_bytes and leaf_info non-NULL; out->steps and a bound observation ring whenever
 * frames are produced (obs or leaf_rows).  Issued on `stream` (the engine's step stream): one launch, plus the raster
 * kernel and the root-frame copy with frames, plus the row writer with leaf rows. */
typedef struct {
  const cbev_snapshot_info* src_info; /* NULL: roots are live env ids (as cbev_lookahead)                 */
  const void* src_rows;               /* rows of src_info, 16-byte aligned                                 */
  const int32_t* roots;               /* [B] env ids or row ids, NULL = identity (B <= N / n_rows)         */
  void* obs;                          /* nullable: leaf windows [B][F][cbev_frame_bytes], 16-byte aligned  */
  int64_t obs_bytes;
  void* leaf_rows;                    /* nullable: B snapshot rows, 16-byte aligned                        */
  int64_t leaf_bytes;
  cbev_snapshot_info* leaf_info;      /* required with leaf_rows                                           */
} cbev_lookahead_io;
int cbev_lookahead_ex(cbev_handle h, const cbev_lookahead_io* io, int32_t n_branches, int32_t horizon,
                      const void* actions_dev, double gamma, const cbev_lookahead_out* out, void* stream);

/* cbev_fuse on n caller-owned windows laid out [n][F][cbev_frame_bytes] (what cbev_lookahead_obs writes) instead of
 * the ring: out_dev gets [n][C-1+3][oh][ow] (VEHICLE_TEMPORAL, the masks' element type) or float32 [n][C][oh][ow]
 * (VEHICLE_WEIGHTED), bit-identical to cbev_fuse of envs holding those windows.  The checks of cbev_fuse (mode,
 * semantic masks with a vehicle channel, frame_stack >= 3), plus non-null 16-byte aligned buffers and n >= 1.  One
 * launch on `stream`; needs no ring and no reset. */
int cbev_fuse_windows(cbev_handle h, int32_t mode, const void* windows_dev, int32_t n, void* out_dev, void* stream);

/* Debug / parity: keep the 128x128 palette-index frame of every env (one extra 16 KB store per env-step
 * while on), and copy the last one out (uint8 [N][S][S], device pointer). */
int cbev_keep_fov(cbev_handle h, int32_t on);
int cbev_copy_fov(cbev_handle h, uint8_t* fov_dev, void* stream);

/* Global episode statistics accumulated on device (CBEV_STATS_FIELDS doubles, device pointer).
 * The caller all-reduces this vector across ranks (NCCL) -- the engine has no other exchange. */
int cbev_read_stats(cbev_handle h, double* stats_dev, int32_t reset_after, void* stream);

/* Number of kernel launches issued by the engine so far. */
int64_t cbev_launch_count(cbev_handle h);

/* Per-kernel device timing: when enabled, cbev_step records CUDA events around its three kernels on the streams
 * they are launched on (k_move and k_render on `stream`, k_judge on the side stream; up to 2048 steps are kept).
 * cbev_profile_read(_ex) synchronises and returns the summed durations in milliseconds (sim_ms = k_move). */
int cbev_profile_enable(cbev_handle h, int32_t on);
int cbev_profile_read(cbev_handle h, double* sim_ms, double* render_ms, int64_t* steps);
int cbev_profile_read_ex(cbev_handle h, double* move_ms, double* render_ms, double* judge_ms, int64_t* steps);

/* Test / measurement hooks (bit values; results are identical).  Any other bit is rejected with CBEV_ERR_ARG.
 *   1   force the generic rotate path (pygame's per-pixel range tests and background colour) even when the window
 *       corners prove it unnecessary -- the reference's crop sizes never need it, so this is the only way to exercise it
 *   2   k_judge serial on the caller's stream instead of the side stream      4  record the per-CTA phase timeline
 *   32  identity CTA -> env order in the raster kernel                       128  identity group -> env order in k_move
 *   256 route size 128 / (96, 96) through k_render_any                       512  k_render_any without its 8:3 block shortcut
 *   1024 the step goes through the fused k_step_repeat (cbev_set_action_repeat) also at repeat 1 */
int cbev_set_debug_flags(cbev_handle h, int32_t flags);

/* Diagnostic: per-CTA phase timestamps of the last raster launch (enable with debug flag 4 before the step).
 * host_out: uint64[N][8] = globaltimer ns at {start, tile landed, draw list done, rotate done, resize done,
 * stores issued}, SM id, unused. */
int cbev_debug_read_trace(cbev_handle h, uint64_t* host_out);

/* ABI self-check: sizeof(cbev_config), sizeof(cbev_pool_desc), sizeof(cbev_step_out). */
int cbev_abi_sizes(int32_t* config_bytes, int32_t* pool_desc_bytes, int32_t* step_out_bytes);

#ifdef __cplusplus
}
#endif
#endif /* CBEV_H */

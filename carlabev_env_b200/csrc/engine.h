// engine.h -- internal layout of the CarlaBEV B200 engine (not part of the C ABI).
//
// HBM layout (all struct-of-arrays):
//   * PoolDev   : read-only scene pool, flat arrays + offset tables (one copy per GPU)
//   * EnvState  : per-env mutable state, env-major; actor arrays are [N][max_actors]
//   * RenderDesc: per-env render descriptor written by the sim kernel, read by the raster kernel
//   * obs ring  : caller-owned, [N][ring_slots][frame]
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/cbev.h"

#define CBEV_TGT_WORDS 2      // 64-bit words of target-visibility bits per env
#define CBEV_MAX_TARGETS (64 * CBEV_TGT_WORDS)  // ego route points (targets) per scene, one visibility bit each
#define CBEV_RECT_WORDS 2     // draw-list entry: x0 | y0 << 16, (w - 1) | (h - 1) << 12 | palette << 24
#define CBEV_DESC_WORDS 20    // ints per render-descriptor header
#define CBEV_TILE_H 184       // rows of the class-map tile one frame can sample (fetch window, sim.cu:compute_view)
#define CBEV_TILE_W 208       // tile pitch in bytes: window (<= 184) + 15 bytes of TMA alignment slack, rounded up to
                              // an ODD number of 16-byte chunks (rows then rotate through the shared-memory banks)
#define CBEV_WARPS_PER_BLOCK 4
#define CBEV_PROF_MAX 2048
#define CBEV_PROF_EVENTS 5     // per profiled step: before k_move, after k_move, after k_render, before / after k_judge

// render descriptor header words
enum {
  RD_OX = 0,   // fetch-window origin in MAP coordinates, may be negative (TMA zero-fills = NON_DRIVABLE)
  RD_OY,
  RD_MODE,     // 0: exact 90-degree turns, 1: 16.16 fixed-point walk
  RD_TURNS,
  RD_NX, RD_NY, RD_ISIN, RD_ICOS, RD_AX, RD_AY, RD_XD, RD_YD, RD_CY,
  RD_NRECTS,
  RD_FLAGS,    // bit0: reset frame (fill every window slot), bit1: skip this env (masked-out env of a partial reset)
  RD_FX, RD_FY,  // fetch-window origin in CROP coordinates (rebases the rotate walk onto the tile)
  RD_BG        // palette index of crop pixel (0, 0) after drawing = transform.rotate's background colour
};

struct EnvState {
  int32_t* scene = nullptr;        // [N] pool index, -1 before the first reset
  int32_t* episode = nullptr;      // [N] episodes finished by this env
  uint8_t* done = nullptr;         // [N] last step was terminal (needs reset)
  double* ego = nullptr;           // [N][24]: x,y,yaw,v,x1,y1,yaw1,v1,acc,t,dist2goal,dist2goal_1,s_prev,last_dyaw,
                                   //          previous comfort (accel_long, accel_lat, yaw_rate), target speed,
                                   //          decoded action + applied steering angle of the step (sim.cu E_*)
  int32_t* egoi = nullptr;         // [N][8]: tidx, flags(bit0 comfort valid, bit1 s_prev valid), k, consecutive_offroad, step
  unsigned long long* tgt_vis = nullptr;  // [N][CBEV_TGT_WORDS]
  double* stats = nullptr;         // [N][12]: return, length, sum speed, sum |comfort| x6, viol, harsh, cause
  // actors [N][max_actors]
  double *ax = nullptr, *ay = nullptr, *ayaw = nullptr, *av = nullptr, *atarget_mps = nullptr;
  double *aelapsed = nullptr, *astate_elapsed = nullptr;
  int32_t *atidx = nullptr, *arxlen = nullptr;
  uint8_t* aflags = nullptr;       // bits0-3 fsm, bit4 braking, bit5 on retreat route
  // retreat routes [N][max_retreat][CBEV_SG_MAX][3] + lengths [N][max_retreat]
  double* retreat = nullptr;
  int32_t* retreat_n = nullptr;
};

// The per-env sections of EnvState after the header (scene, episode, done), in snapshot-row order, with their element
// size and their element count per env (A = max(max_actors, 1) actor slots, R retreat slots).  The one list of what an
// env's state is: snapshot rows (snapshot.cu) and the lookahead branch state (sim.cu, api.cu) are both built from it.
#define CBEV_STATE_SECTIONS 16
struct StateSections {
  void** field[CBEV_STATE_SECTIONS];  // the EnvState member that holds each section's device array
  int32_t esize[CBEV_STATE_SECTIONS], count[CBEV_STATE_SECTIONS];
};
inline StateSections cbev_state_sections(EnvState& st, int32_t A, int32_t R) {
  return StateSections{
      {(void**)&st.ego, (void**)&st.egoi, (void**)&st.tgt_vis, (void**)&st.stats, (void**)&st.ax, (void**)&st.ay,
       (void**)&st.ayaw, (void**)&st.av, (void**)&st.atarget_mps, (void**)&st.aelapsed, (void**)&st.astate_elapsed,
       (void**)&st.atidx, (void**)&st.arxlen, (void**)&st.aflags, (void**)&st.retreat, (void**)&st.retreat_n},
      {8, 4, 8, 8, 8, 8, 8, 8, 8, 8, 8, 4, 4, 1, 8, 4},
      {24, 8, CBEV_TGT_WORDS, 12, A, A, A, A, A, A, A, A, A, A, R * 3 * CBEV_SG_MAX, R}};
}

__device__ __forceinline__ void cbev_copy_elem(uint8_t* d, const uint8_t* s, int es) {
  if (es == 8) *(uint64_t*)d = *(const uint64_t*)s;
  else if (es == 4) *(uint32_t*)d = *(const uint32_t*)s;
  else *d = *s;
}
__device__ __forceinline__ void cbev_zero_elem(uint8_t* d, int es) {
  if (es == 8) *(uint64_t*)d = 0;
  else if (es == 4) *(uint32_t*)d = 0;
  else *d = 0;
}

struct PoolDev {
  int32_t n_scenes = 0, n_actors_total = 0, max_actors = 0, max_targets = 0, max_tl = 0, max_retreat = 0;
  double *ego_state0 = nullptr, *ego_target_speed = nullptr, *len_ego_route = nullptr;
  int32_t *ego_tidx0 = nullptr, *num_vehicles = nullptr;
  int32_t *ego_off = nullptr, *rew_off = nullptr, *actor_off = nullptr, *tl_off = nullptr;
  double *ego_cx = nullptr, *ego_cy = nullptr, *ego_cyaw = nullptr;
  int32_t *rew_rx = nullptr, *rew_ry = nullptr;
  double* rew_cum = nullptr;
  uint8_t *act_kind = nullptr, *act_beh = nullptr;
  double *act_state0 = nullptr, *act_cruise_px = nullptr, *act_cruise_mps = nullptr, *act_beh_p = nullptr;
  int32_t *act_tidx0 = nullptr, *act_route_off = nullptr, *act_raw_off = nullptr;
  int32_t* act_retreat_slot = nullptr;  // per actor: slot in the per-env retreat-route buffer or -1
  double *act_cx = nullptr, *act_cy = nullptr, *act_cyaw = nullptr, *act_raw_x = nullptr, *act_raw_y = nullptr;
  int32_t* tl_rect = nullptr;
  uint8_t* tl_color = nullptr;
  double* sg_mat = nullptr;
  // open-loop actor trajectories: pose after step t of actor a of scene s at traj[traj_off[s] + t * A_s + a]
  int32_t traj_steps = 0;
  double4* traj = nullptr;
  long long* traj_off = nullptr;
  EnvState roll;  // actor state of every scene after traj_steps steps (rows = scenes), continuation for long episodes
};

struct SimParams {
  int32_t N, max_actors, max_rects, max_retreat;
  int32_t map_w, map_h, fov, crop, pad, anchor_x, anchor_y;
  int32_t hero_w, win_max;  // ego square (hero.py:17); largest fetch window the raster kernel holds
  float hero_scale;         // hero.py:14: int(1024 / size)
  int32_t action_mode, n_discrete, reward_mode, autoreset;
  uint64_t seed;
  const uint8_t* map;
  float discrete_table[16 * 3];
  cbev_config cfg;  // reward parameters
};

// ResizeObservation variants (cv2.resize INTER_AREA from the S x S field of view, S = EnvConfig.size)
#define CBEV_RS_FAST96 0  /* 128 -> (96, 96): 4x4-block two-pass kernel, weights in 1/16 (k_render)        */
#define CBEV_RS_TABLE 1   /* shrinking on both axes: OpenCV's float32 area tables                          */
#define CBEV_RS_HALF 2    /* exactly S/2 on both axes: OpenCV's 2x2 fast path, (a + b + c + d + 2) >> 2    */
#define CBEV_RS_COPY 3    /* (S, S): cv2.resize returns a copy                                             */
#define CBEV_RS_LINEAR 4  /* an axis enlarges (size 64 -> 96): OpenCV's 8-bit bilinear kernel on area-mode */
                          /* coefficients (11-bit fixed point)                                             */
#define CBEV_ANY_BOX_W 128  /* k_render_any: the fetch window lands as column strips of 128 bytes (one TMA box each) */

// cbev_set_debug_flags bits (include/cbev.h); only the launchers read them
enum {
  CBEV_DBG_GENERIC_ROTATE = 1,          // generic (range-tested) rotate path even where the window corners prove it unneeded
  CBEV_DBG_JUDGE_SERIAL = 2,            // k_judge on the caller's stream, serial between k_move and k_render
  CBEV_DBG_TRACE = 4,                   // per-CTA phase timeline of the raster kernel (cbev_debug_read_trace)
  CBEV_DBG_IDENTITY_RENDER_ORDER = 32,  // raster CTA b renders env b
  CBEV_DBG_IDENTITY_MOVE_ORDER = 128,   // k_move group g steps env g
  CBEV_DBG_RENDER_ANY = 256,            // size 128 / (96, 96) through k_render_any
  CBEV_DBG_NO_BLOCK83 = 512,            // k_render_any without its 8:3 block shortcut
  CBEV_DBG_STEP_REPEAT = 1024,          // the step goes through k_step_repeat also at action repeat 1
  CBEV_DBG_KNOWN = CBEV_DBG_GENERIC_ROTATE | CBEV_DBG_JUDGE_SERIAL | CBEV_DBG_TRACE | CBEV_DBG_IDENTITY_RENDER_ORDER |
                   CBEV_DBG_IDENTITY_MOVE_ORDER | CBEV_DBG_RENDER_ANY | CBEV_DBG_NO_BLOCK83 | CBEV_DBG_STEP_REPEAT
};

struct cbev_engine {
  cbev_config cfg;
  int device = 0;
  int32_t N = 0, crop = 0, pad = 0, anchor_x = 0, anchor_y = 0;
  int32_t map_w = 0, map_h = 0;
  uint8_t* map = nullptr;
  alignas(64) unsigned char tmap[128];  // CUtensorMap of the class map, box = CBEV_TILE_W x CBEV_TILE_H (k_render)
  alignas(64) unsigned char tmap_any[128];  // same map, box = CBEV_ANY_BOX_W x any_box_h (k_render_any)
  int32_t win_max = 0;                  // largest fetch window (rows / columns) the raster kernel in use can hold
  int32_t any_nbx = 0, any_nby = 0, any_box_h = 0;  // k_render_any: strips x row boxes of the fetch window
  bool has_map = false, has_pool = false, was_reset = false, keep_fov = false;
  PoolDev pool;
  EnvState st;
  int32_t max_rects = 0;
  int32_t debug_flags = 0;         // cbev_set_debug_flags
  int32_t action_repeat = 1;       // cbev_set_action_repeat: simulator steps per step call
  int32_t* desc = nullptr;         // [N][CBEV_DESC_WORDS]
  uint32_t* rects = nullptr;       // [N][max_rects][CBEV_RECT_WORDS]
  int32_t* order = nullptr;        // [N] raster CTA b renders env order[b]: envs that fill the whole frame window (reset
                                   //     frames, F times the stores) first, so they do not form the tail of the launch
  int32_t* order_cnt = nullptr;    // [2] heavy / light counters of the step (zeroed by the raster kernel)
  int32_t* move_order = nullptr;   // [N] group g of k_move steps env move_order[g]: k_judge puts the envs that will
                                   //     auto-reset next step first, so that the (long) reset path and the normal path
                                   //     do not serialise inside the same warps
  int32_t* move_cnt = nullptr;     // [2] counters behind move_order (zeroed by k_move)
  uint8_t* fov = nullptr;          // [N][S][S] last palette-index frame (debug / RGB path)
  unsigned long long* trace = nullptr;  // [N][8] phase timestamps (debug flag 4)
  int32_t rs_mode = 0, rs_words = 0;  // CBEV_RS_*: how ResizeObservation is computed for this obs_size
  int32_t* rs_tab = nullptr;          // device: OpenCV area tables of both axes (generic obs sizes)
  uint8_t* fov_mask = nullptr;     // [S][S] 0x00 / 0xff corner mask (fov_masked) or null
  void* ring = nullptr;
  int64_t ring_bytes = 0, frame_bytes = 0;
  void* final_obs = nullptr;       // caller-owned [N][F][frame_bytes] terminal windows (CBEV_AUTORESET_SAME_STEP) or null
  int32_t channels = 0;
  int32_t head = -1;
  double* gstats = nullptr;        // [CBEV_STATS_FIELDS]
  // staging for cbev_step_host
  void* h_actions_dev = nullptr;
  double* h_reward_dev = nullptr;
  uint8_t *h_term_dev = nullptr, *h_trunc_dev = nullptr;
  // k_judge (reward / termination / statistics) and the D2H copies of cbev_step_host run on a high-priority side
  // stream, overlapped with the raster kernel
  cudaStream_t side_stream = nullptr;
  cudaEvent_t ev_sim = nullptr, ev_copy = nullptr, ev_judge = nullptr;
  bool host_copy_pending = false;           // cbev_wait_host_outputs has something to wait for
  int64_t launches = 0;
  int64_t steps = 0;
  // per-kernel profiling (cbev_profile_enable)
  bool profiling = false;
  cudaEvent_t* prof_ev = nullptr;  // [CBEV_PROF_MAX][CBEV_PROF_EVENTS]
  int32_t prof_n = 0;
  bool prof_fused[CBEV_PROF_MAX] = {};  // profiled step i ran k_step_repeat (no k_judge)
  // snapshot rows (cbev_snapshot / cbev_restore) restore only into this engine and this pool epoch
  uint64_t token = 0;
  int32_t pool_epoch = 0;          // bumped by cbev_invalidate and by every pool upload that does not extend the last
  // lookahead branch state (cbev_lookahead): scene, episode, done + the state sections, branch_rows rows at up to
  // branch_retreat retreat slots; allocated on first use, grown when either is exceeded
  EnvState branch;
  int32_t branch_rows = 0, branch_retreat = 0;
  // leaf windows of cbev_lookahead_ex when the caller asks for leaf rows but not for the windows: [B][F][frame_bytes],
  // allocated on first use, grown when exceeded
  uint8_t* br_window = nullptr;
  int64_t br_window_bytes = 0;
  // branch render state (cbev_lookahead_obs): per-step draw records in staging slot t mod F, and the [B * F] render
  // positions of the leaf windows the raster kernel reads; room for br_rows branches at br_max_rects draw-list entries
  // (the stride: reallocated when a pool upload raises max_rects), allocated on first use, grown when either is
  // exceeded.  A call with B branches uses the first F * B frame slots of each buffer:
  int32_t* br_stage_desc = nullptr;   // [F][B][CBEV_DESC_WORDS]
  uint32_t* br_stage_rects = nullptr; // [F][B][br_max_rects][CBEV_RECT_WORDS]
  int32_t* br_desc = nullptr;         // [B * F][CBEV_DESC_WORDS]
  uint32_t* br_rects = nullptr;       // [B * F][br_max_rects][CBEV_RECT_WORDS]
  int32_t br_rows = 0, br_max_rects = 0;
};

// Snapshot row of one env (snapshot.cu), every section 16-byte aligned, A = max(max_actors, 1), R = retreat slots:
//   0    int32 scene, int32 episode, int32 done, int32 0
//   16   ego      double[24]          208  egoi   int32[8]   240  tgt_vis  uint64[2]   256  stats  double[12]
//   352  ax, ay, ayaw, av, atarget_mps, aelapsed, astate_elapsed: double[A] each, then atidx, arxlen: int32[A] each,
//        then aflags: uint8[A] (each padded to 16 bytes)
//   ...  retreat double[R][3][CBEV_SG_MAX], retreat_n int32[R] (padded)
//   ...  frames: the F frames of the observation window, oldest first, frame_bytes each
// The padding bytes are written as zeros.
struct SnapLayout {
  int64_t off[CBEV_STATE_SECTIONS];  // row offset of each section
  int32_t esize[CBEV_STATE_SECTIONS], count[CBEV_STATE_SECTIONS];  // element size / count per env (row side)
  int64_t frames_off, row_bytes;
};
SnapLayout cbev_snap_layout(const cbev_engine* e, int32_t retreat_slots);
// snapshot rows as lookahead roots (cbev_lookahead_ex): layout at the rows' retreat slots, base, row count
struct RowSource {
  SnapLayout L;
  const void* rows;
  int32_t n_rows;
};

// kernels (sim.cu / render.cu)
void cbev_launch_reset(cbev_engine* e, const uint8_t* mask, const int32_t* scene_ids, cudaStream_t s);
void cbev_launch_move(cbev_engine* e, const void* actions, const cbev_step_out* out, cudaStream_t s);
void cbev_launch_judge(cbev_engine* e, const cbev_step_out* out, cudaStream_t s);
// k_step_repeat: e->action_repeat simulator steps per env with the judging inline, then the raster launch
void cbev_launch_step_repeat(cbev_engine* e, const void* actions, const cbev_step_out* out, cudaStream_t s);
int cbev_launch_render(cbev_engine* e, int32_t head, int32_t mirror, cudaStream_t s);
// CBEV_AUTORESET_SAME_STEP, after the step: the terminal windows of the envs that ended (flags of `out`) into
// e->final_obs, their reset from the pool and reset descriptor headers; skip headers for the rest.  The raster launch
// at the same head that follows renders the reset frames.
void cbev_launch_same_step_reset(cbev_engine* e, const cbev_step_out* out, int32_t head, cudaStream_t s);
void cbev_set_error(const char* fmt, ...);
// temporal fusion of n windows of L frames each whose newest frame is at slot `head` (the ring, or [n][F] windows)
int cbev_launch_fuse(cbev_engine* e, int32_t mode, const void* ring, int32_t n, int32_t L, int32_t head, void* out,
                     cudaStream_t s);
// raster kernels over n = B * F branch render positions into the caller's [B][F] leaf windows
int cbev_launch_render_branches(cbev_engine* e, int32_t n, void* windows, cudaStream_t s);
void cbev_launch_rollout(cbev_engine* e, cudaStream_t s);
void cbev_launch_generate(cbev_engine* e, const PoolDev& pool, const uint8_t* kinds, const int32_t* levels,
                          const long long* seeds, int32_t* attempts, cudaStream_t s);
void cbev_launch_snapshot(cbev_engine* e, const int32_t* env_ids, int32_t n, void* dst, cudaStream_t s);
void cbev_launch_restore(cbev_engine* e, const SnapLayout& L, const void* src, int32_t n_rows, const int32_t* rows,
                         const int32_t* env_ids, int32_t n, cudaStream_t s);
// record: the leaf windows' draw records (cbev_lookahead_obs); src: roots are rows of src (null: live envs); leaf:
// the branch rows keep what a snapshot row holds (cbev_launch_leaf_rows writes them); repeat: sub-steps per action row
// (cbev_lookahead_repeat, k_lookahead_rep; 1 launches the kernels of the other lookahead calls)
void cbev_launch_lookahead(cbev_engine* e, const int32_t* roots, int32_t n_branches, int32_t horizon,
                           const void* actions, double gamma, const cbev_lookahead_out* out, bool record,
                           const RowSource* src, bool leaf, int32_t repeat, cudaStream_t s);
// the frames of the leaf windows older than each branch's first step, from its root's window: the ring of a live root
// or the frame section of a root row (src); zeros for a root outside [0, N) / [0, n_rows) or a row whose scene lies
// outside the pool
void cbev_launch_leaf_window(cbev_engine* e, const int32_t* roots, int32_t n_branches, const int32_t* steps,
                             void* windows, const RowSource* src, cudaStream_t s);
// branch b's leaf as snapshot row b of dst (current layout): header and state from the branch state, frames from the
// leaf window b of `windows`; a branch without a valid root (branch scene -1) leaves its row unwritten
void cbev_launch_leaf_rows(cbev_engine* e, int32_t n_branches, const void* windows, void* dst, cudaStream_t s);

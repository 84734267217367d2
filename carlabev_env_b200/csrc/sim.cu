// sim.cu -- per-env simulation kernels (one warp per environment).
//
// Restates, for the GPU, the reference's per-step path before rendering:
//   decode_action (envs/spaces.py:43-47) -> BaseAgent.physics_step (src/actors/hero.py:88-138)
//   -> Actor.step / behaviours / Controller.control_step (src/actors/actor.py:110-119,
//      src/actors/behavior/*.py, src/control/stanley_controller.py:51-123, src/control/state.py:29-51)
//   -> Scene.collision_check (src/scenes/scene.py:110-140) -> CaRLRewardFn.step / RewardFn.step
//      (src/deeprl/carl_reward_fn.py:149-341, src/deeprl/reward.py:80-278)
//   -> EpisodeStats.step / termination (src/deeprl/stats.py:30-56, envs/carlabev.py:177-185)
// and emits, per env, the render descriptor (crop origin, pygame.transform.rotate parameters and
// the clipped draw list) consumed by render.cu.
//
// Compiled with -fmad=false: the reference evaluates every product and sum separately in IEEE
// double (NumPy / CPython scalars), so no contraction is allowed here.  Lanes of a warp run the
// scalar ego / reward arithmetic redundantly (uniform), and split route points, actors and
// targets between them; collisions and termination are resolved with warp ballots.
#include <limits.h>
#include <math.h>

#include "engine.h"

#ifndef CBEV_SIM_BLOCKS_PER_SM
#define CBEV_SIM_BLOCKS_PER_SM 7  // 7 x 4 warps/SM: 4096 envs fit in one wave on 148 SMs (<= 73 registers)
#endif

namespace {

constexpr double DT = 0.1;                       // stanley_controller.py:22
constexpr double WB = 2.9;                       // stanley_controller.py:29
constexpr double KST = 2.0;                      // stanley_controller.py:20
constexpr double KPS = 1.0;                      // stanley_controller.py:21
constexpr double MPP = 0.3125;                   // 40 / 128, hero.py:67
constexpr double MAX_STEER = 0x1.0c152382d7365p-1;  // np.radians(30.0)
constexpr double PI = 0x1.921fb54442d18p+1;
constexpr double TWO_PI = 0x1.921fb54442d18p+2;
constexpr double HALF_PI = 0x1.921fb54442d18p+0;
constexpr double DEG2RAD = 0x1.1df46a2529d39p-6;  // math.radians
constexpr double RAD2DEG = 0x1.ca5dc1a63c1f8p+5;  // math.degrees
constexpr unsigned FULL = 0xffffffffu;

// ego double slots
enum { E_X = 0, E_Y, E_YAW, E_V, E_X1, E_Y1, E_YAW1, E_V1, E_ACC, E_T, E_D2G, E_D2G1, E_SPREV, E_LAST_DYAW,
       E_PC_AL, E_PC_AT, E_PC_YR, E_TARGET, E_GAS, E_STEER, E_BRAKE, E_DELTA, E_SLOTS = 24 };
enum { I_TIDX = 0, I_FLAGS, I_K, I_OFFROAD, I_STEP, I_SLOTS = 8 };
enum { S_RET = 0, S_LEN, S_SPEED, S_C0, S_VIOL = 9, S_HARSH, S_CAUSE, S_SLOTS = 12 };
enum { FL_COMFORT = 1, FL_SPREV = 2 };
// fsm states (behavior/jaywalk.py)
enum { ST_IDLE = 0, ST_WAITING, ST_ENTERING, ST_YIELDING, ST_CROSSING, ST_STALLED, ST_RETREATING, ST_CLEARED,
       ST_RETREATED };
enum { HIT_NONE = 0, HIT_VEHICLE, HIT_PEDESTRIAN, HIT_TARGET };

__device__ __forceinline__ double clipd(double x, double lo, double hi) { return fmin(fmax(x, lo), hi); }

// control/utils.py:78 -- NumPy floor-mod
__device__ __forceinline__ double angle_mod(double x) {
  double a = x + PI;
  double m = fmod(a, TWO_PI);
  if (m != 0.0) {
    if (m < 0.0) m += TWO_PI;
  } else {
    m = 0.0;
  }
  return m - PI;
}

__device__ __forceinline__ int rect_left(double c, int pad, int size) {
  // transforms.py:46-51: round(origin + c) with Python banker's rounding, then Rect.center setter
  return (int)rint((double)pad + c * 1.0) - (size >> 1);
}

__device__ __forceinline__ bool overlap(int ax, int ay, int aw, int bx, int by, int bw) {
  return ax < bx + bw && ay < by + bw && ax + aw > bx && ay + aw > by;
}

__device__ __forceinline__ uint64_t splitmix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// calc_target_index (stanley_controller.py:100-117): global argmin of the front-axle distance,
// first minimum wins.  Warp-cooperative; returns the same idx in every lane.
template <int G>
__device__ int warp_nearest(double fx, double fy, const double* __restrict__ cx, const double* __restrict__ cy, int n,
                            int lane, unsigned GM) {
  double best = INFINITY;
  int bi = 0x7fffffff;
  for (int i = lane; i < n; i += G) {
    double dx = fx - cx[i], dy = fy - cy[i];
    double d = dx * dx + dy * dy;
    if (d < best) { best = d; bi = i; }
  }
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) {
    double ob = __shfl_xor_sync(GM, best, o);
    int oi = __shfl_xor_sync(GM, bi, o);
    if (ob < best || (ob == best && oi < bi)) { best = ob; bi = oi; }
  }
  return bi;
}

// scalar version (used inside divergent per-actor code)
__device__ int scalar_nearest(double fx, double fy, const double* cx, const double* cy, int n) {
  double best = INFINITY;
  int bi = 0;
  for (int i = 0; i < n; ++i) {
    double dx = fx - cx[i], dy = fy - cy[i];
    double d = dx * dx + dy * dy;
    if (d < best) { best = d; bi = i; }
  }
  return bi;
}

struct Body {
  double x, y, yaw, v, x1, y1, yaw1, v1;
};

// State.update, state.py:29-51
__device__ __forceinline__ void body_update(Body& b, double acc, double delta, double target) {
  delta = clipd(delta, -MAX_STEER, MAX_STEER);
  b.x1 = b.x; b.y1 = b.y; b.yaw1 = b.yaw; b.v1 = b.v;
  double sn, cs;
  sincos(b.yaw, &sn, &cs);
  b.x += (b.v * cs) * DT;
  b.y += (b.v * sn) * DT;
  b.yaw += ((b.v / WB) * tan(delta)) * DT;
  b.v += acc * DT;
  b.yaw = angle_mod(b.yaw);
  b.v = clipd(b.v, -1.0 * target, target);
}

// ---- render descriptor -------------------------------------------------------------------------
// Camera + pygame.transform.rotate parameters of one frame, and the FETCH WINDOW: the bounding box (in crop
// coordinates) of the source texels the 128 x 128 view can sample.  The view is an affine image of a 128-px square,
// so whatever the crop size (182 px for the centred camera, 230 px for lookahead_75, up to 360 px for a corner
// anchor) the box is at most ceil(128 * sqrt(2)) + 2 = 183 px on a side: the raster kernel fetches a constant
// CBEV_TILE_H x CBEV_TILE_W tile for every configuration.
struct View {
  int xmin, ymin;  // crop origin on the padded scene surface
  int mode, turns, nx, ny, isin, icos, ax, ay, xd, yd, cy;
  int fx, fy, bw, bh;  // fetch window inside the crop
};

__device__ void compute_view(const SimParams& P, double x, double y, double theta, View& v) {
  // Follow.scroll + compute_crop_rect: camera.py:39-42, world.py:105-111, fov.py:70-79
  const int crop = P.crop, pad = P.pad;
  int offx = (int)(((double)pad + x * 1.0) + (-(double)crop / 2.0));
  int offy = (int)(((double)pad + y * 1.0) + (-(double)crop / 2.0));
  int cx = (int)rint((double)offx + (double)crop / 2.0);
  int cy = (int)rint((double)offy + (double)crop / 2.0);
  v.xmin = max(0, min(max(0, P.map_w + 2 * pad - crop), cx - crop / 2));
  v.ymin = max(0, min(max(0, P.map_h + 2 * pad - crop), cy - crop / 2));
  // pygame.transform.rotate(crop, degrees(yaw) + 90): fov.py:84-88, SURVEY.md A.6
  float anglef = (float)(theta * RAD2DEG + 90.0);
  double angle = (double)anglef;
  if (fmod(angle, 90.0) == 0.0) {
    int a = (int)angle;
    int turns = (a / 90) % 4;
    if (turns < 0) turns += 4;
    v.mode = 0;
    v.turns = turns;
    v.nx = v.ny = crop;
    v.isin = v.icos = v.ax = v.ay = v.xd = v.yd = v.cy = 0;
  } else {
    double rad = angle * 0.01745329251994329;
    double s = sin(rad), c = cos(rad);
    double w = (double)crop, h = (double)crop;
    double cxx = c * w, cyy = c * h, sx = s * w, sy = s * h;
    int nx = (int)fmax(fmax(fmax(fabs(cxx + sy), fabs(cxx - sy)), fabs(-cxx + sy)), fabs(-cxx - sy));
    int ny = (int)fmax(fmax(fmax(fabs(sx + cyy), fabs(sx - cyy)), fabs(-sx + cyy)), fabs(-sx - cyy));
    v.mode = 1;
    v.turns = 0;
    v.nx = nx;
    v.ny = ny;
    v.isin = (int)(s * 65536.0);
    v.icos = (int)(c * 65536.0);
    v.ax = (nx << 15) - (int)(c * (double)((nx - 1) << 15));
    v.ay = (ny << 15) - (int)(s * (double)((nx - 1) << 15));
    v.xd = (crop - nx) * 32768;
    v.yd = (crop - ny) * 32768;
    v.cy = ny / 2;
  }
  // fetch window: source texel of the four corners of the view (the map view -> source is affine, floor is monotone)
  const int S = P.fov;
  const int left = P.anchor_x - (v.nx >> 1), top = P.anchor_y - (v.ny >> 1);  // get_rect(center=anchor), fov.py:88-94
  int x_lo = INT_MAX, x_hi = INT_MIN, y_lo = INT_MAX, y_hi = INT_MIN;
#pragma unroll
  for (int c4 = 0; c4 < 4; ++c4) {
    const int rxp = ((c4 & 1) ? S - 1 : 0) - left, ryp = ((c4 & 2) ? S - 1 : 0) - top;
    int sx, sy;
    if (v.mode == 0) {
      if (v.turns == 0) { sx = rxp; sy = ryp; }
      else if (v.turns == 1) { sx = crop - 1 - ryp; sy = rxp; }
      else if (v.turns == 2) { sx = crop - 1 - rxp; sy = crop - 1 - ryp; }
      else { sx = ryp; sy = crop - 1 - rxp; }
    } else {
      sx = ((v.ax + v.xd) + v.isin * (v.cy - ryp) + rxp * v.icos) >> 16;
      sy = ((v.ay + v.yd) - v.icos * (v.cy - ryp) + rxp * v.isin) >> 16;
    }
    x_lo = min(x_lo, sx); x_hi = max(x_hi, sx);
    y_lo = min(y_lo, sy); y_hi = max(y_hi, sy);
  }
  x_lo = max(x_lo, 0); y_lo = max(y_lo, 0);
  x_hi = min(x_hi, crop - 1); y_hi = min(y_hi, crop - 1);
  if (x_hi < x_lo || y_hi < y_lo) { x_lo = y_lo = 0; x_hi = y_hi = 0; }  // the view misses the crop: nothing is sampled
  v.fx = x_lo;
  v.fy = y_lo;
  v.bw = min(x_hi - x_lo + 1, P.win_max);  // <= ceil(S * sqrt(2)) + 2 by the bound above (183 at size 128)
  v.bh = min(y_hi - y_lo + 1, P.win_max);
}

__device__ void write_desc_header(const SimParams& P, int32_t* __restrict__ d, const View& v, int nrects, int flags,
                                  int bg) {
  d[RD_OX] = v.xmin + v.fx - P.pad;  // fetch-window origin in MAP coordinates (may be negative: TMA zero-fills)
  d[RD_OY] = v.ymin + v.fy - P.pad;
  d[RD_MODE] = v.mode;
  d[RD_TURNS] = v.turns;
  d[RD_NX] = v.nx;
  d[RD_NY] = v.ny;
  d[RD_ISIN] = v.isin;
  d[RD_ICOS] = v.icos;
  d[RD_AX] = v.ax;
  d[RD_AY] = v.ay;
  d[RD_XD] = v.xd;
  d[RD_YD] = v.yd;
  d[RD_CY] = v.cy;
  d[RD_NRECTS] = nrects;
  d[RD_FLAGS] = flags;
  d[RD_FX] = v.fx;
  d[RD_FY] = v.fy;
  d[RD_BG] = bg;
}

// palette index of crop pixel (0, 0) of the bare map: transform.rotate's background colour is the source surface's
// first pixel (SURVEY.md A.6); rectangles drawn over it are accounted for by the caller
__device__ __forceinline__ int crop_corner_class(const SimParams& P, const View& v) {
  const int mx = v.xmin - P.pad, my = v.ymin - P.pad;
  if (mx < 0 || my < 0 || mx >= P.map_w || my >= P.map_h) return CBEV_PAL_NON_DRIVABLE;  // padding colour
  return P.map[(size_t)my * P.map_w + mx];
}

// clip a scene-surface rect to the fetch window and pack it (CBEV_RECT_WORDS = 2 words:
// x0 | y0 << 16, (w - 1) | (h - 1) << 12 | palette << 24, window coordinates); returns false if nothing is left.
// `covers00` reports whether the rect covers crop pixel (0, 0), the rotate background sample.
__device__ __forceinline__ bool pack_rect(int rx, int ry, int rw, int rh, int pal, const View& v, uint32_t& w0,
                                          uint32_t& w1, bool& covers00) {
  covers00 = rx <= v.xmin && v.xmin < rx + rw && ry <= v.ymin && v.ymin < ry + rh;
  const int wx = v.xmin + v.fx, wy = v.ymin + v.fy;
  int x0 = max(rx - wx, 0), y0 = max(ry - wy, 0);
  int x1 = min(rx + rw - wx, v.bw), y1 = min(ry + rh - wy, v.bh);
  if (x1 <= x0 || y1 <= y0) return false;
  w0 = (uint32_t)x0 | ((uint32_t)y0 << 16);
  w1 = (uint32_t)(x1 - x0 - 1) | ((uint32_t)(y1 - y0 - 1) << 12) | ((uint32_t)pal << 24);
  return true;
}

// Actor.reset (actors/actor.py:86-108) for every actor of `scene` into row `row` of the actor arrays of S
__device__ void init_actors(const SimParams& P, const PoolDev& pool, const EnvState& S, size_t row, int scene, int lane,
                            int stride) {
  const int A0 = pool.actor_off[scene], A = pool.actor_off[scene + 1] - A0;
  for (int a = lane; a < A; a += stride) {
    size_t o = row * P.max_actors + a;
    const double* s0 = pool.act_state0 + (size_t)(A0 + a) * 4;
    S.ax[o] = s0[0];
    S.ay[o] = s0[1];
    S.ayaw[o] = s0[2];
    S.av[o] = s0[3];
    S.atidx[o] = pool.act_tidx0[A0 + a];
    int beh = pool.act_beh[A0 + a];
    bool jay = beh == CBEV_BEH_CROSS || beh == CBEV_BEH_STOP_MID || beh == CBEV_BEH_STOP_RETURN;
    S.atarget_mps[o] = jay ? 0.0 : pool.act_cruise_mps[A0 + a];  // jaywalk.py:23-28 / actor.py:94-95
    S.aelapsed[o] = 0.0;
    S.astate_elapsed[o] = 0.0;
    S.arxlen[o] = pool.act_raw_off[A0 + a + 1] - pool.act_raw_off[A0 + a];
    S.aflags[o] = jay ? ST_WAITING : ST_IDLE;
  }
}

// ---- reset ------------------------------------------------------------------------------------
// CarlaBEV.reset with a pool scene: Scene.load_scene / reset_all / reward_fn.reset / stats.reset
// (scenes/scene.py:41-88, actors/actor.py:86-108, carl_reward_fn.py:121-134, stats.py:104-105)
__device__ void reset_env(const SimParams& P, const PoolDev& pool, const EnvState& st, int env, int scene, int lane,
                          int stride = 32) {
  const int r0 = pool.ego_off[scene], nt = pool.ego_off[scene + 1] - r0;
  if (lane == 0) {
    double* e = st.ego + (size_t)env * E_SLOTS;
    const double* s0 = pool.ego_state0 + (size_t)scene * 4;
    e[E_X] = e[E_X1] = s0[0];
    e[E_Y] = e[E_Y1] = s0[1];
    e[E_YAW] = e[E_YAW1] = s0[2];
    e[E_V] = e[E_V1] = s0[3];
    e[E_ACC] = 0.0;
    e[E_T] = 0.0;
    double gx = pool.ego_cx[r0 + nt - 1], gy = pool.ego_cy[r0 + nt - 1];
    double dx = s0[0] - gx, dy = s0[1] - gy;
    double d2g = sqrt(dx * dx + dy * dy);  // scene.py:49-52
    e[E_D2G] = e[E_D2G1] = d2g;
    e[E_SPREV] = 0.0;
    e[E_LAST_DYAW] = 0.0;
    e[E_PC_AL] = e[E_PC_AT] = e[E_PC_YR] = 0.0;
    e[E_TARGET] = pool.ego_target_speed[scene];
    int32_t* ei = st.egoi + (size_t)env * I_SLOTS;
    ei[I_TIDX] = pool.ego_tidx0[scene];
    ei[I_FLAGS] = 0;
    ei[I_K] = 0;
    ei[I_OFFROAD] = 0;
    ei[I_STEP] = 0;
    st.scene[env] = scene;
    st.done[env] = 0;
    for (int w = 0; w < CBEV_TGT_WORDS; ++w) {
      const int n = nt - 64 * w;
      st.tgt_vis[(size_t)env * CBEV_TGT_WORDS + w] = n >= 64 ? ~0ull : (n > 0 ? ((1ull << n) - 1ull) : 0ull);
    }
    double* sa = st.stats + (size_t)env * S_SLOTS;
    for (int k = 0; k < S_SLOTS; ++k) sa[k] = 0.0;
  }
  init_actors(P, pool, st, (size_t)env, scene, lane, stride);
}

__global__ void __launch_bounds__(32 * CBEV_WARPS_PER_BLOCK)
k_reset(SimParams P, PoolDev pool, EnvState st, const uint8_t* __restrict__ mask,
        const int32_t* __restrict__ scene_ids, int32_t* __restrict__ desc, int32_t* __restrict__ order,
        int32_t* __restrict__ move_order) {
  const int env = blockIdx.x * CBEV_WARPS_PER_BLOCK + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (env >= P.N) return;
  if (lane == 0) { order[env] = env; move_order[env] = env; }
  if (mask != nullptr && mask[env] == 0) {
    if (lane == 0) desc[(size_t)env * CBEV_DESC_WORDS + RD_FLAGS] = 2;  // bit1: skip rendering this env
    return;
  }
  int scene = scene_ids[env];
  scene = min(max(scene, 0), pool.n_scenes - 1);
  reset_env(P, pool, st, env, scene, lane);
  if (lane == 0) {
    const double* s0 = pool.ego_state0 + (size_t)scene * 4;
    // BaseMap.reset draws the bare map with _theta = 0.0 and no actors (world.py:92-100)
    View v;
    compute_view(P, s0[0], s0[1], 0.0, v);
    write_desc_header(P, desc + (size_t)env * CBEV_DESC_WORDS, v, 0, 1, crop_corner_class(P, v));
  }
}

// ---- mid-episode retreat route (jaywalk.py:43-54 -> stanley_controller.py:34-49 -> utils.py:200-269)
__device__ void start_retreat(const PoolDev& pool, double* rbuf, int32_t* rn, int ga, Body& b, int& tidx, int& rxlen) {
  const int w0 = pool.act_raw_off[ga];
  const double* rawx = pool.act_raw_x + w0;
  const double* rawy = pool.act_raw_y + w0;
  int cur = max(0, min(tidx, rxlen - 1));
  double ax[CBEV_SG_MAX], ay[CBEV_SG_MAX];
  int n0 = min(cur + 2, CBEV_SG_MAX);
  ax[0] = b.x;
  ay[0] = b.y;
  for (int i = 1; i < n0; ++i) {
    ax[i] = rawx[cur - (i - 1)];
    ay[i] = rawy[cur - (i - 1)];
  }
  // drop consecutive duplicates
  int n = 1;
  for (int i = 1; i < n0; ++i) {
    double d = hypot(ax[i] - ax[i - 1], ay[i] - ay[i - 1]);
    if (d > 1e-9) { ax[n] = ax[i]; ay[n] = ay[i]; ++n; }
  }
  if (n < 2) { ax[1] = ax[0] + 1e-3; ay[1] = ay[0]; n = 2; }
  double* cx = rbuf;
  double* cy = rbuf + CBEV_SG_MAX;
  double* cyaw = rbuf + 2 * CBEV_SG_MAX;
  const double* M = pool.sg_mat + (size_t)n * CBEV_SG_MAX * CBEV_SG_MAX;
  for (int i = 0; i < n; ++i) {
    double sx = 0.0, sy = 0.0;
    for (int j = 0; j < n; ++j) {
      sx += M[i * CBEV_SG_MAX + j] * ax[j];
      sy += M[i * CBEV_SG_MAX + j] * ay[j];
    }
    cx[i] = sx;
    cy[i] = sy;
  }
  double s[CBEV_SG_MAX];
  s[0] = 0.0;
  for (int i = 1; i < n; ++i) s[i] = s[i - 1] + hypot(cx[i] - cx[i - 1], cy[i] - cy[i - 1]);
  if (s[n - 1] <= 1e-9) {
    for (int i = 0; i < n; ++i) cyaw[i] = 0.0;
  } else {
    // np.gradient (second order interior, first order edges) + np.arctan2 + np.unwrap
    double prev = 0.0, corr = 0.0;
    for (int i = 0; i < n; ++i) {
      double gx, gy;
      if (i == 0) {
        gx = (cx[1] - cx[0]) / (s[1] - s[0]);
        gy = (cy[1] - cy[0]) / (s[1] - s[0]);
      } else if (i == n - 1) {
        gx = (cx[n - 1] - cx[n - 2]) / (s[n - 1] - s[n - 2]);
        gy = (cy[n - 1] - cy[n - 2]) / (s[n - 1] - s[n - 2]);
      } else {
        double d1 = s[i] - s[i - 1], d2 = s[i + 1] - s[i];
        double a = -(d2) / (d1 * (d1 + d2)), bb = (d2 - d1) / (d1 * d2), c = d1 / (d2 * (d1 + d2));
        gx = a * cx[i - 1] + bb * cx[i] + c * cx[i + 1];
        gy = a * cy[i - 1] + bb * cy[i] + c * cy[i + 1];
      }
      double p = atan2(gy, gx);
      if (i > 0) {
        double dd = p - prev;
        double m = fmod(dd + PI, TWO_PI);
        if (m != 0.0 && m < 0.0) m += TWO_PI;
        double ddmod = m - PI;
        if (ddmod == -PI && dd > 0.0) ddmod = PI;
        double pc = ddmod - dd;
        if (fabs(dd) < PI) pc = 0.0;
        corr += pc;
      }
      prev = p;
      cyaw[i] = i > 0 ? p + corr : p;
    }
  }
  *rn = n;
  // Controller.set_route(jitter_start=False)
  b.x = cx[0];
  b.y = cy[0];
  double fx = b.x + WB * cos(b.yaw), fy = b.y + WB * sin(b.yaw);
  tidx = scalar_nearest(fx, fy, cx, cy, n);
  b.yaw = cyaw[tidx];
  rxlen = cur + 2;
}

// One chunk of G actors of one scene instance: behaviour FSM (Actor.step, actors/actor.py:110-116), Stanley / P
// control with the cooperative nearest-waypoint argmin and the bicycle update (stanley_controller.py:51-123).
// Actor state lives in row `row` of the actor arrays of S (an environment, or a scene during the roll-out).
// Returns the post-step pose in `b` and the actor kind.
template <int G>
__device__ __forceinline__ void actor_chunk_step(const SimParams& P, const PoolDev& pool, const EnvState& S, size_t row,
                                                 int ga, size_t o, bool has, double t_sim, int lane, int gb, unsigned GM,
                                                 Body& b, int& kind) {
    int atidx = 0, rxlen = 0, fsm = 0, np = 0, beh = 0;
    kind = 0;
    bool braking = false, on_retreat = false;
    double target_mps = 0.0, elapsed = 0.0, state_elapsed = 0.0, cruise_mps = 0.0;
    const double *cxp = nullptr, *cyp = nullptr, *cyawp = nullptr;
    double* rbuf = nullptr;
    int32_t* rnp = nullptr;
    if (has) {
      b.x = S.ax[o]; b.y = S.ay[o]; b.yaw = S.ayaw[o]; b.v = S.av[o];
      b.x1 = b.x; b.y1 = b.y; b.yaw1 = b.yaw; b.v1 = b.v;
      atidx = S.atidx[o];
      rxlen = S.arxlen[o];
      int fl = S.aflags[o];
      fsm = fl & 15; braking = fl & 16; on_retreat = fl & 32;
      target_mps = S.atarget_mps[o];
      kind = pool.act_kind[ga];
      beh = pool.act_beh[ga];
      cruise_mps = pool.act_cruise_mps[ga];
      int slot = pool.act_retreat_slot ? pool.act_retreat_slot[ga] : -1;
      if (slot >= 0) {
        rbuf = S.retreat + (row * P.max_retreat + slot) * (3 * CBEV_SG_MAX);
        rnp = S.retreat_n + row * P.max_retreat + slot;
      }
      if (on_retreat) {
        cxp = rbuf; cyp = rbuf + CBEV_SG_MAX; cyawp = rbuf + 2 * CBEV_SG_MAX; np = *rnp;
      } else {
        int ro = pool.act_route_off[ga];
        np = pool.act_route_off[ga + 1] - ro;
        cxp = pool.act_cx + ro; cyp = pool.act_cy + ro; cyawp = pool.act_cyaw + ro;
      }
      // ---- behaviour (Actor.step: behaviour first, actor.py:110-116) ----
      if (beh == CBEV_BEH_LEAD_BRAKE) {  // lead_brake.py:10-15
        const double* p = pool.act_beh_p + (size_t)ga * 4;
        if (t_sim >= p[0]) braking = true;
        if (braking) target_mps = fmax(0.0, target_mps - p[1] * DT);
      } else if (beh != CBEV_BEH_NONE) {  // jaywalk.py:56-138
        const double* p = pool.act_beh_p + (size_t)ga * 4;
        elapsed = S.aelapsed[o] + DT;
        state_elapsed = S.astate_elapsed[o] + DT;
        const bool complete = atidx >= rxlen - 1;
        if (beh == CBEV_BEH_CROSS) {
          if (fsm == ST_WAITING) {
            target_mps = 0.0;
            if (elapsed >= p[0]) { fsm = ST_CROSSING; state_elapsed = 0.0; target_mps = fmax(0.0, cruise_mps); }
          } else if (fsm == ST_CROSSING) {
            target_mps = fmax(0.0, cruise_mps);
            if (complete) { fsm = ST_CLEARED; state_elapsed = 0.0; target_mps = 0.0; }
          } else if (fsm == ST_CLEARED) {
            target_mps = 0.0;
          }
        } else {
          const bool has_stop = p[2] >= 0.0;
          const bool retreat = p[3] != 0.0;
          if (fsm == ST_WAITING) {
            target_mps = 0.0;
            if (elapsed >= p[0]) { fsm = ST_ENTERING; state_elapsed = 0.0; target_mps = fmax(0.0, cruise_mps); }
          } else if (fsm == ST_ENTERING) {
            target_mps = fmax(0.0, cruise_mps);
            int mid = max(1, min(rxlen - 1, (int)(p[1] * (double)(rxlen - 1))));
            if (atidx >= mid) {
              fsm = (retreat || has_stop) ? ST_YIELDING : ST_STALLED;
              state_elapsed = 0.0; target_mps = 0.0;
            } else if (complete) {
              fsm = ST_CLEARED; state_elapsed = 0.0; target_mps = 0.0;
            }
          } else if (fsm == ST_YIELDING) {
            target_mps = 0.0;
            if (has_stop && state_elapsed >= p[2]) {
              if (retreat && rbuf != nullptr && pool.sg_mat != nullptr) {
                start_retreat(pool, rbuf, rnp, ga, b, atidx, rxlen);
                on_retreat = true;
                cxp = rbuf; cyp = rbuf + CBEV_SG_MAX; cyawp = rbuf + 2 * CBEV_SG_MAX; np = *rnp;
                fsm = ST_RETREATING; state_elapsed = 0.0; target_mps = fmax(0.0, cruise_mps);
              } else {
                fsm = ST_CROSSING; state_elapsed = 0.0; target_mps = fmax(0.0, cruise_mps);
              }
            }
          } else if (fsm == ST_CROSSING) {
            target_mps = fmax(0.0, cruise_mps);
            if (complete) { fsm = ST_CLEARED; state_elapsed = 0.0; target_mps = 0.0; }
          } else if (fsm == ST_STALLED) {
            target_mps = 0.0;
          } else if (fsm == ST_RETREATING) {
            target_mps = fmax(0.0, cruise_mps);
            int w0 = pool.act_raw_off[ga];
            double gx = b.x - pool.act_raw_x[w0], gy = b.y - pool.act_raw_y[w0];
            bool reached = sqrt(gx * gx + gy * gy) <= 1.0;
            if (reached || complete) { fsm = ST_RETREATED; state_elapsed = 0.0; target_mps = 0.0; }
          } else if (fsm == ST_CLEARED || fsm == ST_RETREATED) {
            target_mps = 0.0;
          }
        }
      }
    }
    // ---- Controller.control_step (stanley_controller.py:51-62): frozen once at the last waypoint
    const bool active = has && (atidx < np - 1);
    double fx = 0.0, fy = 0.0;
    if (active) {
      double sn, cs;
      sincos(b.yaw, &sn, &cs);
      fx = b.x + WB * cs; fy = b.y + WB * sn;
    }
    int my_idx = 0;
    unsigned am = __ballot_sync(GM, active) >> gb;
    while (am) {
      int src = __ffs(am) - 1;
      am &= am - 1;
      double bfx = __shfl_sync(GM, fx, gb + src), bfy = __shfl_sync(GM, fy, gb + src);
      unsigned long long pcx = __shfl_sync(GM, (unsigned long long)cxp, gb + src);
      unsigned long long pcy = __shfl_sync(GM, (unsigned long long)cyp, gb + src);
      int bn = __shfl_sync(GM, np, gb + src);
      int idx = warp_nearest<G>(bfx, bfy, (const double*)pcx, (const double*)pcy, bn, lane, GM);
      if (lane == src) my_idx = idx;
    }
    if (active) {
      const double target = target_mps / MPP;  // set_target_speed_mps, actor.py:121-124
      double ai = KPS * (target - b.v);
      double ddx = fx - cxp[my_idx], ddy = fy - cyp[my_idx];
      double sn2, cs2;
      sincos(b.yaw + HALF_PI, &sn2, &cs2);
      double err = ddx * (-cs2) + ddy * (-sn2);  // stanley_controller.py:119-121
      int cur = atidx >= my_idx ? atidx : my_idx;
      double theta_e = angle_mod(cyawp[cur] - b.yaw);
      double theta_d = atan2(KST * err, fmax(b.v, 1e-3));
      double di = clipd(theta_e + theta_d, -MAX_STEER, MAX_STEER);
      atidx = cur;
      body_update(b, ai, di, target);
    }
    if (has) {
      S.ax[o] = b.x; S.ay[o] = b.y; S.ayaw[o] = b.yaw; S.av[o] = b.v;
      S.atidx[o] = atidx;
      S.arxlen[o] = rxlen;
      S.atarget_mps[o] = target_mps;
      S.aelapsed[o] = elapsed;
      S.astate_elapsed[o] = state_elapsed;
      S.aflags[o] = (uint8_t)(fsm | (braking ? 16 : 0) | (on_retreat ? 32 : 0));
    }
}

// Cold paths of k_move.  Keeping them OUT of line (to shrink the hot instruction stream: ncu round 2 shows "no
// instruction" as the second stall reason of the 7.6 k-instruction kernel) was measured on B200 and is much slower --
// k_move 17 -> 29 us at 4096 envs: the call ABI forces the live values of the caller through local memory -- so they
// are inlined.
template <int G>
__device__ __forceinline__ void live_actor_chunk(const SimParams& P, const PoolDev& pool, const EnvState& S, size_t row, int ga,
                                              size_t o, bool has, double t_sim, int lane, int gb, unsigned GM, Body& b,
                                              int& kind) {
  actor_chunk_step<G>(P, pool, S, row, ga, o, has, t_sim, lane, gb, GM, b, kind);
}

template <int G>
__device__ __forceinline__ void hand_over_to_live(const SimParams& P, const PoolDev& pool, const EnvState& st, int env, int scene,
                                               int A, int lane, unsigned GM) {
  for (int a = lane; a < A; a += G) {
    const size_t o = (size_t)env * P.max_actors + a, r = (size_t)scene * P.max_actors + a;
    st.ax[o] = pool.roll.ax[r]; st.ay[o] = pool.roll.ay[r]; st.ayaw[o] = pool.roll.ayaw[r]; st.av[o] = pool.roll.av[r];
    st.atarget_mps[o] = pool.roll.atarget_mps[r]; st.aelapsed[o] = pool.roll.aelapsed[r];
    st.astate_elapsed[o] = pool.roll.astate_elapsed[r]; st.atidx[o] = pool.roll.atidx[r];
    st.arxlen[o] = pool.roll.arxlen[r]; st.aflags[o] = pool.roll.aflags[r];
  }
  for (int k = lane; k < P.max_retreat * 3 * CBEV_SG_MAX; k += G)
    st.retreat[(size_t)env * P.max_retreat * 3 * CBEV_SG_MAX + k] = pool.roll.retreat[(size_t)scene * P.max_retreat * 3 * CBEV_SG_MAX + k];
  for (int k = lane; k < P.max_retreat; k += G)
    st.retreat_n[(size_t)env * P.max_retreat + k] = pool.roll.retreat_n[(size_t)scene * P.max_retreat + k];
  __syncwarp(GM);
}

// The pool scene of an env's device auto-reset: a hash of (seed, env, episodes finished), shared by both auto-reset
// modes so that SAME_STEP draws at the terminal call the scene NEXT_STEP draws at the call after it.
__device__ __forceinline__ int auto_reset_scene(const SimParams& P, const PoolDev& pool, const EnvState& st, int env) {
  int ep = st.episode[env];
  uint64_t h = splitmix64(P.seed + (uint64_t)env * 0x9E3779B97F4A7C15ull + (uint64_t)ep * 0xD1B54A32D192ED03ull);
  return (int)(h % (uint64_t)pool.n_scenes);
}

template <int G>
__device__ __forceinline__ void auto_reset_env(const SimParams& P, const PoolDev& pool, const EnvState& st, const cbev_step_out& out,
                                            int32_t* d, int32_t* order, int32_t* order_cnt, int env, int lane, unsigned GM) {
  int scene = auto_reset_scene(P, pool, st, env);
  __syncwarp(GM);
  reset_env(P, pool, st, env, scene, lane, G);
  if (lane == 0) {
    order[atomicAdd(order_cnt, 1)] = env;  // heavy: the reset frame goes to all F window slots -> rendered first
    const double* s0 = pool.ego_state0 + (size_t)scene * 4;
    View v;
    compute_view(P, s0[0], s0[1], 0.0, v);
    write_desc_header(P, d, v, 0, 1, crop_corner_class(P, v));  // bit0: reset frame; k_judge skips this env
    out.reward[env] = 0.0;
    out.terminated[env] = 0;
    out.truncated[env] = 0;
    if (out.cause) out.cause[env] = CBEV_CAUSE_NONE;
    if (out.hero) {
      double* hb = out.hero + (size_t)env * CBEV_HERO_FIELDS;
      for (int k = 0; k < CBEV_HERO_FIELDS; ++k) hb[k] = 0.0;
      hb[CBEV_H_X] = s0[0]; hb[CBEV_H_Y] = s0[1]; hb[CBEV_H_YAW] = s0[2]; hb[CBEV_H_V] = s0[3];
      hb[CBEV_H_SCENE] = (double)scene;
    }
  }
}

// ---- the step kernels ---------------------------------------------------------------------------
// The step is split where the reference's data flow allows it (envs/carlabev.py:223-231, scenes/scene.py:90-140):
//   k_move  -- everything that MOVES: action decode, ego bicycle physics, scripted actors (trajectory tables or live
//              behaviour FSM + Stanley), and what the rasteriser needs from it: the crop / rotate descriptor and the
//              clipped draw list.  Short dependent chain; the raster kernel waits only for this.
//   k_judge -- everything that JUDGES the new state: nearest waypoint, comfort signals, rect collisions / proximity /
//              TTC, target consumption, tile lookup, CaRL / shaping reward, termination, episode statistics, info
//              block.  The long fp64 chain; runs on a side stream CONCURRENTLY with the raster kernel, which reads
//              only the descriptor and the draw list.
// G lanes cooperate on one environment (32 / G environments per warp).  The scalar arithmetic runs uniformly on the
// G lanes of a group, so a smaller G wastes less of the fp64 pipe; G = 32 is used when scenes carry many actors that
// are stepped live (lanes = actors), G = 8 otherwise.
template <int G>
struct Group {
  int warp, lane, gb, grp;
  unsigned GM;
  int env;
  __device__ __forceinline__ Group(const SimParams& P, const int32_t* __restrict__ perm = nullptr) {
    constexpr int EPW = 32 / G;
    warp = threadIdx.x >> 5;
    const int wl = threadIdx.x & 31;
    lane = wl & (G - 1);   // lane within the environment's group
    gb = wl & ~(G - 1);    // first warp lane of the group
    grp = wl / G;
    GM = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << gb);
    env = (blockIdx.x * CBEV_WARPS_PER_BLOCK + warp) * EPW + grp;
    if (perm != nullptr && env < P.N) env = perm[env];
  }
};

// The bodies of k_move and k_judge are shared with k_lookahead.  The branch instantiations (MV_BRANCH, and judge_body's
// BRANCH = true) step row `env` of a private branch state and leave out everything only the live step needs -- the
// view, draw list and render descriptor, the CTA and move orders, the episode statistics (per-env accumulators, episode
// block, gstats, st.episode / st.done) and auto-reset.  What remains is the same code, so a branch step is
// bit-identical to a live step of the same state with the same action.  MV_BRANCH_DRAW (k_lookahead_obs) also keeps
// the view, the draw list and the descriptor header, written at `env` of the caller's `desc` / `rects` (a staging slot
// of the branch render state), but no CTA order: the frame it describes is then bit-identical to the live one.
enum { MV_LIVE = 0, MV_BRANCH = 1, MV_BRANCH_DRAW = 2 };
template <int G, int MODE>
__device__ __forceinline__ void move_body(const SimParams& P, const PoolDev& pool, const EnvState& st,
                                          const void* __restrict__ actions, const cbev_step_out& out,
                                          int32_t* __restrict__ desc, uint32_t* __restrict__ rects,
                                          int32_t* __restrict__ order, int32_t* __restrict__ order_cnt, int env,
                                          int lane, int gb, unsigned GM) {
  constexpr bool BRANCH = MODE != MV_LIVE, DRAW = MODE != MV_BRANCH;
  int32_t* d = desc + (size_t)env * CBEV_DESC_WORDS;
  uint32_t* rl = rects + (size_t)env * P.max_rects * CBEV_RECT_WORDS;

  // First level of loads, all independent of each other and issued together (the kernel is a chain of dependent
  // global loads, ~0.7 us each under load: done -> scene -> offsets -> table): the done flag, the scene index, the
  // ego state and the action.  An env that auto-resets simply does not use them.
  const uint8_t was_done = BRANCH ? 0 : st.done[env];
  const int scene = st.scene[env];
  double* eg = st.ego + (size_t)env * E_SLOTS;
  const int32_t* ei = st.egoi + (size_t)env * I_SLOTS;
  Body e;
  e.x = eg[E_X]; e.y = eg[E_Y]; e.yaw = eg[E_YAW]; e.v = eg[E_V];
  double acc = eg[E_ACC];
  const double etarget = eg[E_TARGET];
  const double t_sim = eg[E_T] + DT;  // scene.py:91 (k_judge stores it)
  const int step_idx = ei[I_STEP];
  const unsigned long long tv0 = st.tgt_vis[(size_t)env * CBEV_TGT_WORDS], tv1 = st.tgt_vis[(size_t)env * CBEV_TGT_WORDS + 1];
  // ---- a1: decode action (spaces.py:43-47, hero.py:165-187) ----------------------------------------
  float gas, steer, brake;
  if (P.action_mode == CBEV_ACTION_DISCRETE) {
    long long id = ((const long long*)actions)[env];
    const int nd = P.n_discrete;
    id = id < 0 ? 0 : (id >= nd ? nd - 1 : id);
    gas = P.discrete_table[id * 3 + 0];
    steer = P.discrete_table[id * 3 + 1];
    brake = P.discrete_table[id * 3 + 2];
  } else {
    const float* a = (const float*)actions + (size_t)env * 3;
    gas = fminf(fmaxf(a[0], 0.0f), 1.0f);
    steer = fminf(fmaxf(a[1], -1.0f), 1.0f);
    brake = fminf(fmaxf(a[2], 0.0f), 1.0f);
  }

  // ---- device auto-reset (gymnasium NEXT_STEP semantics) from the pool -------------------------
  if constexpr (!BRANCH) {
    if (P.autoreset == CBEV_AUTORESET_NEXT_STEP && was_done) {
      auto_reset_env<G>(P, pool, st, out, d, order, order_cnt, env, lane, GM);
      return;
    }
  }

  // second level: everything that depends only on the scene index
  const int r0 = pool.ego_off[scene], nt = pool.ego_off[scene + 1] - r0;
  const int A0 = pool.actor_off[scene], A = pool.actor_off[scene + 1] - A0;
  const int tl0 = pool.tl_off[scene], ntl = pool.tl_off[scene + 1] - tl0;
  const bool use_table = step_idx < pool.traj_steps;
  const long long toff = pool.traj_steps > 0 ? pool.traj_off[scene] : 0;
  const double* __restrict__ ecx = pool.ego_cx + r0;
  const double* __restrict__ ecy = pool.ego_cy + r0;

  // ---- a2/a3: ego physics (uniform across lanes) ------------------------------------------------
  double acc_val = gas > 0.0f ? (double)__fmul_rn(gas, P.hero_scale) : 0.0;  // hero.py:14,142: 8 at size 128
  double delta;
  if (fabs(e.v) < 0.1) {
    delta = 0.0;
  } else {
    double steer_deg = clipd(18.0 / (1.0 + 0.35 * fabs(e.v)), 8.0, 18.0);
    delta = ((double)steer * steer_deg) * DEG2RAD;
  }
  double speed_factor = clipd(fabs(e.v) / 5.0, 0.3, 1.0);
  double brake_val = (brake > 0.0f ? (double)__fmul_rn(__fmul_rn(brake, 0.6f), P.hero_scale) : 0.0) * speed_factor;
  double target_acc = acc_val - brake_val - 0.05 * e.v;
  acc = (1.0 - 0.2) * acc + 0.2 * target_acc;
  const double applied_delta = delta;
  body_update(e, acc, delta, etarget);
  e.v *= 0.9999;
  if (fabs(e.v) < 0.05) e.v = 0.0;
  e.v *= 0.985;
  if (lane == 0) {
    eg[E_X] = e.x; eg[E_Y] = e.y; eg[E_YAW] = e.yaw; eg[E_V] = e.v;
    eg[E_X1] = e.x1; eg[E_Y1] = e.y1; eg[E_YAW1] = e.yaw1; eg[E_V1] = e.v1;
    eg[E_ACC] = acc;
    eg[E_GAS] = (double)gas; eg[E_STEER] = (double)steer; eg[E_BRAKE] = (double)brake; eg[E_DELTA] = applied_delta;
  }

  const int pad = P.pad;
  View view;
  int bg = 0;
  if constexpr (DRAW) {
    compute_view(P, e.x, e.y, e.yaw, view);
    bg = crop_corner_class(P, view);  // rotate background: crop pixel (0, 0) after every draw below
  }

  // ---- a4/a5: scripted actors ---------------------------------------------------------------------
  // Scripted actors never read the ego (SURVEY.md A.3): their trajectories are functions of (scene, step).
  // The first traj_steps steps of every scene were rolled out at pool upload by the same device code
  // (k_rollout); afterwards the env continues live from the roll-out's final state.
  int nrects = 0;
  if (!use_table && pool.traj_steps > 0 && step_idx == pool.traj_steps) hand_over_to_live<G>(P, pool, st, env, scene, A, lane, GM);
  // table look-ups are software-pipelined: the pose and kind of the next chunk of G actors are fetched while the
  // current chunk is clipped and packed (50-vehicle scenes take 7 chunks at G = 8)
  double4 qn = make_double4(0.0, 0.0, 0.0, 0.0);
  int kn = 0;
  if (use_table && lane < A) {
    qn = pool.traj[toff + (size_t)step_idx * A + lane];
    kn = pool.act_kind[A0 + lane];
  }
  for (int base = 0; base < A; base += G) {
    const int a = base + lane;
    const bool has = a < A;
    const int ga = A0 + (has ? a : 0);
    const size_t o = (size_t)env * P.max_actors + (has ? a : 0);
    Body b;
    int kind = 0;
    if (use_table) {
      const double4 q = qn;
      kind = kn;
      if (a + G < A) {
        qn = pool.traj[toff + (size_t)step_idx * A + a + G];
        kn = pool.act_kind[ga + G];
      }
      if (has) {  // open-loop actors: pose after this step was rolled out once per scene at pool upload
        b.x = q.x; b.y = q.y; b.yaw = q.z; b.v = q.w;
        st.ax[o] = b.x; st.ay[o] = b.y; st.ayaw[o] = b.yaw; st.av[o] = b.v;  // read back by k_judge / cbev_get_state
      }
    } else {
      live_actor_chunk<G>(P, pool, st, (size_t)env, ga, o, has, t_sim, lane, gb, GM, b, kind);
    }
    if constexpr (!DRAW) continue;  // the rest of the chunk draws
    // ---- a6: draw list (vehicles then pedestrians; pool stores them in that order) ----
    const int size = kind == 0 ? 4 : 2;  // vehicle.py:24, pedestrian.py:24
    uint32_t pk0 = 0, pk1 = 0;
    bool vis = false, c00 = false;
    const int pal = kind == 0 ? CBEV_PAL_VEHICLE : CBEV_PAL_PEDESTRIAN;
    if (has) {
      const int rx = rect_left(b.x, pad, size), ry = rect_left(b.y, pad, size);
      vis = pack_rect(rx, ry, size, size, pal, view, pk0, pk1, c00);
    }
    {
      unsigned bm = __ballot_sync(GM, c00) >> gb;
      if (bm) bg = __shfl_sync(GM, pal, gb + 31 - __clz(bm));  // the last rect drawn over the corner wins
    }
    unsigned vm = __ballot_sync(GM, vis) >> gb;
    if (vis) {
      uint32_t* w = rl + (size_t)(nrects + __popc(vm & ((1u << lane) - 1u))) * CBEV_RECT_WORDS;
      w[0] = pk0; w[1] = pk1;
    }
    nrects += __popc(vm);
  }
  if constexpr (DRAW) {  // the rest only draws
    // ---- targets still visible at draw time (target.py:46-50); k_judge consumes them afterwards ----------
    for (int base = 0; base < nt; base += G) {
      int i = base + lane;
      bool has = i < nt && ((((i >> 6) ? tv1 : tv0) >> (i & 63)) & 1ull);
      int size = (i == nt - 1) ? 4 : 2;  // scenes/utils.py:114-122
      uint32_t pk0 = 0, pk1 = 0;
      bool vis = false, c00 = false;
      if (has) {
        const int tx = rect_left(ecx[i], pad, size), ty = rect_left(ecy[i], pad, size);
        vis = pack_rect(tx, ty, size, size, CBEV_PAL_ROUTE, view, pk0, pk1, c00);
      }
      if (__ballot_sync(GM, c00)) bg = CBEV_PAL_ROUTE;
      unsigned vm = __ballot_sync(GM, vis) >> gb;
      if (vis) {
        uint32_t* w = rl + (size_t)(nrects + __popc(vm & ((1u << lane) - 1u))) * CBEV_RECT_WORDS;
        w[0] = pk0; w[1] = pk1;
      }
      nrects += __popc(vm);
    }
    // ---- traffic lights: drawn without the padding offset (traffic_light.py:81-90, quirk C-4) ----------
    {
      const int t0 = tl0;
      for (int base = 0; base < ntl; base += G) {
        int i = base + lane;
        uint32_t pk0 = 0, pk1 = 0;
        bool vis = false, c00 = false;
        int pal = 0;
        if (i < ntl) {
          const int32_t* r = pool.tl_rect + (size_t)(t0 + i) * 4;
          pal = pool.tl_color[t0 + i];
          vis = pack_rect(r[0], r[1], r[2], r[3], pal, view, pk0, pk1, c00);
        }
        {
          unsigned bm = __ballot_sync(GM, c00) >> gb;
          if (bm) bg = __shfl_sync(GM, pal, gb + 31 - __clz(bm));
        }
        unsigned vm = __ballot_sync(GM, vis) >> gb;
        if (vis) {
          uint32_t* w = rl + (size_t)(nrects + __popc(vm & ((1u << lane) - 1u))) * CBEV_RECT_WORDS;
          w[0] = pk0; w[1] = pk1;
        }
        nrects += __popc(vm);
      }
    }
    if (lane == 0) {
      write_desc_header(P, d, view, nrects, 0, bg);
      if constexpr (!BRANCH) order[P.N - 1 - atomicAdd(order_cnt + 1, 1)] = env;  // light: one frame
    }
  }
}

template <int G>
__global__ void __launch_bounds__(32 * CBEV_WARPS_PER_BLOCK, G == 32 ? CBEV_SIM_BLOCKS_PER_SM : 4)
k_move(SimParams P, PoolDev pool, EnvState st, const void* __restrict__ actions, cbev_step_out out,
       int32_t* __restrict__ desc, uint32_t* __restrict__ rects, int32_t* __restrict__ order,
       int32_t* __restrict__ order_cnt, const int32_t* __restrict__ move_order, int32_t* __restrict__ move_cnt) {
  const Group<G> g(P, move_order);
  if (blockIdx.x == 0 && threadIdx.x < 2 && move_cnt != nullptr) move_cnt[threadIdx.x] = 0;  // k_judge counts afresh
  if (g.env >= P.N) return;
  move_body<G, MV_LIVE>(P, pool, st, actions, out, desc, rects, order, order_cnt, g.env, g.lane, g.gb, g.GM);
}

// 128 registers (4 blocks per SM).  A 64-register variant (8 blocks per SM, 256 B of spills) was measured beside the
// raster kernel: it runs 91 instead of 72 us and the step gets SLOWER (0.1955 vs 0.1919 ms at 4096 envs) -- what the
// raster kernel loses to k_judge grows with the time k_judge stays resident, not with the registers it holds.
// `hb_s` is the group's hero block in shared memory.  The live step writes its outputs at `env`; a branch step
// (JG_BRANCH, JG_BRANCH_ROW) returns reward, flags and cause to the caller, and writes the hero block at `env` only
// when `last` or the step is terminal.  JG_BRANCH_ROW (branches whose leaf becomes a snapshot row) also keeps the
// per-env episode accumulators and the terminal bookkeeping of st.episode / st.done, but not the episode block, the
// gstats atomics or the move order: its row then holds what the live step would have left there.  JG_LIVE_REPEAT
// (k_step_repeat) is JG_LIVE without the move-order writes, and writes the hero block only when `last` or the step is
// terminal.
enum { JG_LIVE = 0, JG_BRANCH = 1, JG_BRANCH_ROW = 2, JG_LIVE_REPEAT = 3 };
template <int G, int MODE>
__device__ __forceinline__ void judge_body(const SimParams& P, const PoolDev& pool, const EnvState& st,
                                           const cbev_step_out& out, double* __restrict__ gstats,
                                           int32_t* __restrict__ move_order, int32_t* __restrict__ move_cnt,
                                           double* __restrict__ hb_s, int env, int lane, int gb, unsigned GM, bool last,
                                           double& reward_out, bool& terminated_out, bool& truncated_out,
                                           int& cause_out) {
  constexpr bool BRANCH = MODE == JG_BRANCH || MODE == JG_BRANCH_ROW;
  const int scene = st.scene[env];
  const int r0 = pool.ego_off[scene], nt = pool.ego_off[scene + 1] - r0;
  const double* __restrict__ ecx = pool.ego_cx + r0;
  const double* __restrict__ ecy = pool.ego_cy + r0;
  const double* __restrict__ ecyaw = pool.ego_cyaw + r0;
  double* eg = st.ego + (size_t)env * E_SLOTS;
  int32_t* ei = st.egoi + (size_t)env * I_SLOTS;

  // the pose k_move produced, and the one before it
  Body e;
  e.x = eg[E_X]; e.y = eg[E_Y]; e.yaw = eg[E_YAW]; e.v = eg[E_V];
  e.x1 = eg[E_X1]; e.y1 = eg[E_Y1]; e.yaw1 = eg[E_YAW1]; e.v1 = eg[E_V1];
  const double acc = eg[E_ACC];
  const double t_sim = eg[E_T] + DT;  // scene.py:91
  int tidx = ei[I_TIDX];
  int flags = ei[I_FLAGS];
  {  // Controller.calc_target_index on the pre-step pose (hero.py:100-104, stanley_controller.py:76-77)
    double sn, cs;
    sincos(e.yaw1, &sn, &cs);
    int idx = warp_nearest<G>(e.x1 + WB * cs, e.y1 + WB * sn, ecx, ecy, nt, lane, GM);
    if (tidx < idx) tidx = idx;
  }
  // compute_comfort_kinematics, comfort.py:17-61
  double speed_mps = e.v * MPP, prev_speed_mps = e.v1 * MPP;
  double dyaw_c = e.yaw - e.yaw1;
  double yaw_rate_rad = atan2(sin(dyaw_c), cos(dyaw_c)) / DT;
  double yaw_rate_deg = yaw_rate_rad * RAD2DEG;
  double accel_long = (speed_mps - prev_speed_mps) / DT;
  double accel_lat = speed_mps * yaw_rate_rad;
  double jerk_long = 0.0, jerk_lat = 0.0, yaw_acc = 0.0;
  if (flags & FL_COMFORT) {
    jerk_long = (accel_long - eg[E_PC_AL]) / DT;
    jerk_lat = (accel_lat - eg[E_PC_AT]) / DT;
    yaw_acc = (yaw_rate_deg - eg[E_PC_YR]) / DT;
  }
  flags |= FL_COMFORT;

  // ego rect (hero.sync_rect, hero.py:34-35)
  const int pad = P.pad;
  const int hw = P.hero_w;  // hero.py:17: int(32 / scale), 4 px at size 128
  const int hx = rect_left(e.x, pad, hw), hy = rect_left(e.y, pad, hw);
  const int hcx = hx + (hw >> 1), hcy = hy + (hw >> 1);

  // ---- a9: collision / proximity (scene.py:110-140, actor.py:166-176) on the actor poses of this step ----
  const int A0 = pool.actor_off[scene], A = pool.actor_off[scene + 1] - A0;
  int hit = HIT_NONE, hit_id = -1, n_nearby = 0;
  double min_ttc = INFINITY;
  double hvx_m, hvy_m, hvx, hvy;
  {
    double sn, cs;
    sincos(e.yaw, &sn, &cs);
    hvx = e.v * cs; hvy = e.v * sn;                 // compute_ttc (px units)
    hvx_m = (e.v * MPP) * cs; hvy_m = (e.v * MPP) * sn;  // compute_ttc_raw (metres)
  }
  for (int base = 0; base < A; base += G) {
    const int a = base + lane;
    const bool has = a < A;
    const size_t o = (size_t)env * P.max_actors + (has ? a : 0);
    int kind = 0, rx = 0, ry = 0;
    bool near = false, coll = false;
    if (has) {
      kind = pool.act_kind[A0 + a];
      const int size = kind == 0 ? 4 : 2;  // vehicle.py:24, pedestrian.py:24
      rx = rect_left(st.ax[o], pad, size);
      ry = rect_left(st.ay[o], pad, size);
      int dcx = hcx - (rx + (size >> 1)), dcy = hcy - (ry + (size >> 1));
      near = dcx * dcx + dcy * dcy < 35 * 35;  // math.hypot(ints) < min_dist
      coll = overlap(hx, hy, hw, rx, ry, size);
    }
    unsigned cm = __ballot_sync(GM, coll) >> gb;
    if (cm) {
      int src = 31 - __clz(cm);  // last colliding actor in iteration order wins
      int k = __shfl_sync(GM, kind, gb + src);
      hit = k == 0 ? HIT_VEHICLE : HIT_PEDESTRIAN;
      hit_id = k;  // Actor.id: Vehicle passes id=0, Pedestrian id=1 (vehicle.py:23, pedestrian.py:23)
    }
    n_nearby += __popc(__ballot_sync(GM, near));
    if (near) {
      const double bx = st.ax[o], by = st.ay[o], byaw = st.ayaw[o], bv = st.av[o];
      double sn, cs;
      sincos(byaw, &sn, &cs);
      double avx = bv * cs, avy = bv * sn;
      double rxx, ryy, rvx, rvy;
      if (P.reward_mode == CBEV_REWARD_CARL) {  // compute_ttc_raw, reward_signals.py:45-94
        rxx = bx * MPP - e.x * MPP; ryy = by * MPP - e.y * MPP;
        rvx = avx * MPP - hvx_m; rvy = avy * MPP - hvy_m;
      } else {                                  // compute_ttc, reward_signals.py:15-42
        rxx = bx - e.x; ryy = by - e.y;
        rvx = avx - hvx; rvy = avy - hvy;
      }
      double nrm = sqrt(rxx * rxx + ryy * ryy);
      double rel = (rvx * rxx + rvy * ryy) / (nrm + 1e-6);
      if (rel < 0.0) min_ttc = fmin(min_ttc, fabs(nrm / rel));
    }
  }
#pragma unroll
  for (int o2 = G / 2; o2 > 0; o2 >>= 1) min_ttc = fmin(min_ttc, __shfl_xor_sync(GM, min_ttc, o2));

  // ---- targets: consumed on overlap, last in order wins (target.py:37-44) ----------------
  unsigned long long tvis[CBEV_TGT_WORDS];
#pragma unroll
  for (int w = 0; w < CBEV_TGT_WORDS; ++w) tvis[w] = st.tgt_vis[(size_t)env * CBEV_TGT_WORDS + w];
  for (int base = 0; base < nt; base += G) {
    int i = base + lane;
    bool has = i < nt && ((tvis[(i >> 6) & (CBEV_TGT_WORDS - 1)] >> (i & 63)) & 1ull);
    int size = (i == nt - 1) ? 4 : 2;  // scenes/utils.py:114-122
    bool coll = false;
    if (has) {
      const int tx = rect_left(ecx[i], pad, size), ty = rect_left(ecy[i], pad, size);
      coll = overlap(hx, hy, hw, tx, ty, size);
    }
    unsigned cm = __ballot_sync(GM, coll) >> gb;
    if (cm) {
      tvis[(base >> 6) & (CBEV_TGT_WORDS - 1)] &= ~((unsigned long long)cm << (base & 63));
      hit = HIT_TARGET;
      hit_id = base + 31 - __clz(cm);
    }
  }

  // ---- dist2goal bookkeeping (scene.py:97-98) ----
  double d2g_1 = eg[E_D2G];
  double d2g;
  {
    double dx = e.x - ecx[nt - 1], dy = e.y - ecy[nt - 1];
    d2g = sqrt(dx * dx + dy * dy);
  }
  // ---- a8: semantic tile under the ego (world.py:159-165) ----
  int tile;
  {
    int txi = (int)clipd(rint(e.x), 0.0, (double)(P.map_w - 1));
    int tyi = (int)clipd(rint(e.y), 0.0, (double)(P.map_h - 1));
    tile = P.map[(size_t)tyi * P.map_w + txi];
  }
  // controller_info (stanley_controller.py:140-176)
  double dist2wp;
  {
    double dx = e.x - ecx[tidx], dy = e.y - ecy[tidx];
    dist2wp = sqrt(dx * dx + dy * dy);
  }
  int w_lo = tidx, w_n = (tidx + 5 <= nt) ? 5 : max(nt - 1 - tidx, 0);  // next_wps(5)

  // lateral_error(signed=True), control/utils.py:165-197
  double lat_err = INFINITY;
  for (int i = 0; i + 1 < w_n; ++i) {
    double Ax = ecx[w_lo + i], Ay = ecy[w_lo + i], Bx = ecx[w_lo + i + 1], By = ecy[w_lo + i + 1];
    double ABx = Bx - Ax, ABy = By - Ay, APx = e.x - Ax, APy = e.y - Ay;
    double tt = (APx * ABx + APy * ABy) / (ABx * ABx + ABy * ABy);
    tt = clipd(tt, 0.0, 1.0);
    double qx = e.x - (Ax + tt * ABx), qy = e.y - (Ay + tt * ABy);
    double er = sqrt(qx * qx + qy * qy);
    double cross = ABx * APy - ABy * APx;
    if (cross != 0.0) er *= (cross > 0.0 ? 1.0 : -1.0);
    if (fabs(er) < fabs(lat_err)) lat_err = er;
  }

  int viol = (fabs(accel_long) > 2.0) + (fabs(accel_lat) > 2.0) + (fabs(yaw_rate_deg) > 20.0) +
             (fabs(jerk_long) > 3.0) + (fabs(jerk_lat) > 3.0) + (fabs(yaw_acc) > 120.0);  // comfort.py:3-10,64-70

  // ---- a10/a11: reward ----
  const cbev_config& C = P.cfg;
  double reward = 0.0;
  int cause = CBEV_CAUSE_NONE;
  double s_prev = eg[E_SPREV], last_dyaw = eg[E_LAST_DYAW];
  int kcount = ei[I_K], offroad = ei[I_OFFROAD];
  const bool goal_hit = hit == HIT_TARGET && hit_id == nt - 1;
  if (P.reward_mode == CBEV_REWARD_CARL) {
    if (tile == CBEV_PAL_NON_DRIVABLE) { reward = -1.0; cause = CBEV_CAUSE_COLLISION; }
    else if (goal_hit) { reward = 1.0; cause = CBEV_CAUSE_SUCCESS; }
    else if (hit == HIT_TARGET) { reward = 0.1; cause = CBEV_CAUSE_CKPT; }
    else if (hit != HIT_NONE) { reward = -1.0; cause = CBEV_CAUSE_COLLISION; }
    else if (dist2wp > 50.0) { reward = -1.0; cause = CBEV_CAUSE_OUT_OF_BOUNDS; }
    else {
      // compute_route_progress, carl_reward_fn.py:29-58 (first closest segment wins)
      const int q0 = pool.rew_off[scene], nq = pool.rew_off[scene + 1] - q0;
      const int32_t* qx = pool.rew_rx + q0;
      const int32_t* qy = pool.rew_ry + q0;
      const double* qc = pool.rew_cum + q0;
      double best = 1e9;
      int bi = 0x7fffffff;
      for (int i = lane; i + 1 < nq; i += G) {
        double Ax = qx[i], Ay = qy[i];
        int abx = qx[i + 1] - qx[i], aby = qy[i + 1] - qy[i];
        double tt = ((e.x - Ax) * (double)abx + (e.y - Ay) * (double)aby) / ((double)(abx * abx + aby * aby) + 1e-9);
        tt = clipd(tt, 0.0, 1.0);
        double px = e.x - (Ax + tt * (double)abx), py = e.y - (Ay + tt * (double)aby);
        double dist = sqrt(px * px + py * py);
        if (dist < best) { best = dist; bi = i; }
      }
#pragma unroll
      for (int o2 = G / 2; o2 > 0; o2 >>= 1) {
        double ob = __shfl_xor_sync(GM, best, o2);
        int oi = __shfl_xor_sync(GM, bi, o2);
        if (ob < best || (ob == best && oi < bi)) { best = ob; bi = oi; }
      }
      double s_t = 0.0;
      if (bi != 0x7fffffff) {
        double Ax = qx[bi], Ay = qy[bi];
        int abx = qx[bi + 1] - qx[bi], aby = qy[bi + 1] - qy[bi];
        double tt = ((e.x - Ax) * (double)abx + (e.y - Ay) * (double)aby) / ((double)(abx * abx + aby * aby) + 1e-9);
        tt = clipd(tt, 0.0, 1.0);
        s_t = qc[bi] + tt * sqrt((double)(abx * abx + aby * aby));
      }
      if (!(flags & FL_SPREV)) { s_prev = s_t; flags |= FL_SPREV; }
      double rc_raw = fmax(0.0, s_t - s_prev);
      s_prev = s_t;
      double total = nq > 0 ? qc[nq - 1] : 0.0;
      double rc = total > 0.0 ? rc_raw / total : 0.0;
      rc = clipd(rc * 100.0, 0.0, 1.0);
      double dist_m = fabs(lat_err) * MPP;
      double ratio = dist_m / 3.0;
      if (C.lane_center_exponent != 1.0) ratio = pow(ratio, C.lane_center_exponent);
      double p_route = dist_m <= 0.0 ? 1.0 : fmax(C.lane_center_floor, 1.0 - ratio);
      bool off_lane = (tile == CBEV_PAL_SIDEWALK) || (dist_m > 1.5 * 3.0);
      double p_off = off_lane ? C.off_lane_penalty : 1.0;
      double over = fmax(speed_mps - 35.0 / 3.6, 0.0);
      double p_speed = over <= 0.0 ? 1.0 : fmax(C.speed_penalty_floor, exp(-over / C.speed_penalty_scale));
      double p_ttc = fmax(C.ttc_penalty_floor, min_ttc < C.ttc_threshold ? 0.5 : 1.0);
      double p_comfort = viol > 0 ? 1.0 - 0.5 * ((double)viol / 6.0) : 1.0;
      double Pt = 1.0;
      Pt *= p_route; Pt *= p_off; Pt *= p_speed; Pt *= p_ttc; Pt *= p_comfort;
      reward = clipd(rc * Pt, 0.0, 1.0);
    }
  } else {
    kcount += 1;
    reward = -0.002;
    if (kcount >= C.max_actions) { reward = 0.0; cause = CBEV_CAUSE_MAX_ACTIONS; }
    else if (dist2wp > 60.0) { reward = -1.0; cause = CBEV_CAUSE_OUT_OF_BOUNDS; }
    else if (tile == CBEV_PAL_NON_DRIVABLE) { reward = -1.0; cause = CBEV_CAUSE_COLLISION; }
    else if (hit == HIT_PEDESTRIAN) { reward = -20.0; cause = CBEV_CAUSE_COLLISION; }
    else if (hit == HIT_VEHICLE) { reward = -12.0; cause = CBEV_CAUSE_COLLISION; }
    else if (goal_hit) { reward = 18.0; cause = CBEV_CAUSE_SUCCESS; }
    else if (hit == HIT_TARGET) { reward = 0.7; cause = CBEV_CAUSE_CKPT; }
    else {
      bool on_sidewalk = tile == CBEV_PAL_SIDEWALK;
      if (on_sidewalk) {
        offroad += 1;
        reward += C.sidewalk_step_penalty + C.sidewalk_penalty_scale * (double)offroad;
      } else {
        offroad = 0;
      }
      if (C.offroad_terminate_after && offroad >= C.offroad_terminate_after) {
        reward -= 0.7;
        cause = CBEV_CAUSE_OFF_ROAD;
      } else {  // RewardFn.non_terminal, reward.py:166-265
        double r = 0.0;
        double desired = ecyaw[tidx];
        double yaw_error = atan2(sin(desired - e.yaw), cos(desired - e.yaw));
        double align = cos(yaw_error);
        double ee = clipd(fabs(lat_err), 0.0, C.lat_clip);
        r -= C.k_lat_quadratic * (ee * ee);
        if (dist2wp > C.route_dev_start) r -= C.k_route_dev * (dist2wp - C.route_dev_start);
        double dprog = d2g_1 - d2g;
        if (dprog > 0.0 && !on_sidewalk) r += (C.k_progress * dprog) * fmax(0.0, align);
        if (e.v > 0.3 && !on_sidewalk) r += (C.k_flow * fmin(e.v, C.max_speed_for_flow)) * fmax(0.0, align);
        if (ee < C.lat_small && fabs(yaw_error) < C.yaw_small) r += C.k_align_bonus;
        double ttc_term = min_ttc < INFINITY ? -exp(-min_ttc / 30.0) : 0.0;
        r += C.k_ttc * ttc_term;
        if (e.v < -0.1) r += -C.k_reverse * fabs(e.v);
        double dyaw = e.yaw1 - e.yaw;
        double steer_jerk = fabs(dyaw - last_dyaw);
        last_dyaw = dyaw;
        r -= C.k_steer_smooth * fabs(dyaw);
        r -= C.k_steer_jerk * steer_jerk;
        r += -C.k_smooth * (fabs(e.v1 - e.v) + fabs(dyaw));
        r += C.alive_bias;
        reward += tanh(r * 1.2);
      }
      reward = clipd(reward, -1.0, 1.0);
    }
  }
  const bool terminated = cause == CBEV_CAUSE_COLLISION || cause == CBEV_CAUSE_SUCCESS ||
                          cause == CBEV_CAUSE_OUT_OF_BOUNDS || cause == CBEV_CAUSE_OFF_ROAD ||
                          cause == CBEV_CAUSE_MAX_ACTIONS;  // carlabev.py:177-185
  const bool truncated = cause == CBEV_CAUSE_MAX_ACTIONS;
  const bool hero_now = out.hero != nullptr && (MODE == JG_LIVE || last || terminated || truncated);

  // ---- a13: episode statistics (stats.py:30-56) ----
  double* sa = st.stats + (size_t)env * S_SLOTS;
  double ep_ret = sa[S_RET] + reward, ep_len = sa[S_LEN] + 1.0, ep_speed = sa[S_SPEED] + e.v;
  double cm6[6] = {fabs(accel_long), fabs(accel_lat), fabs(jerk_long), fabs(jerk_lat), fabs(yaw_rate_deg),
                   fabs(yaw_acc)};
  double ep_viol = sa[S_VIOL] + (viol > 0 ? 1.0 : 0.0);
  double ep_harsh = sa[S_HARSH] + (accel_long < -2.0 ? 1.0 : 0.0);
  double ep_cause = cause != CBEV_CAUSE_NONE ? (double)cause : sa[S_CAUSE];

  // ---- write back (lane 0) ----
  if (lane == 0) {
    eg[E_T] = t_sim; eg[E_D2G] = d2g; eg[E_D2G1] = d2g_1;  // the pose itself was stored by k_move
    eg[E_SPREV] = s_prev; eg[E_LAST_DYAW] = last_dyaw;
    eg[E_PC_AL] = accel_long; eg[E_PC_AT] = accel_lat; eg[E_PC_YR] = yaw_rate_deg;
    ei[I_TIDX] = tidx; ei[I_FLAGS] = flags; ei[I_K] = kcount; ei[I_OFFROAD] = offroad; ei[I_STEP] += 1;
#pragma unroll
    for (int w = 0; w < CBEV_TGT_WORDS; ++w) st.tgt_vis[(size_t)env * CBEV_TGT_WORDS + w] = tvis[w];
    if constexpr (MODE == JG_BRANCH_ROW) {
      if (terminated) {
        st.episode[env] += 1;
        st.done[env] = 1;
        for (int k = 0; k < S_SLOTS; ++k) sa[k] = 0.0;
      } else {
        sa[S_RET] = ep_ret; sa[S_LEN] = ep_len; sa[S_SPEED] = ep_speed;
        for (int k = 0; k < 6; ++k) sa[S_C0 + k] += cm6[k];
        sa[S_VIOL] = ep_viol; sa[S_HARSH] = ep_harsh; sa[S_CAUSE] = ep_cause;
      }
    }
    if constexpr (!BRANCH) {
      out.reward[env] = reward;
      out.terminated[env] = terminated;
      out.truncated[env] = truncated;
      if (out.cause) out.cause[env] = (uint8_t)cause;
      if (terminated) {
        double inv = 1.0 / ep_len;
        if (out.episode) {
          double* ep = out.episode + (size_t)env * CBEV_EPISODE_FIELDS;
          ep[CBEV_E_RETURN] = ep_ret; ep[CBEV_E_LENGTH] = ep_len; ep[CBEV_E_CAUSE] = ep_cause;
          ep[CBEV_E_MEAN_SPEED] = ep_speed / ep_len;
          for (int k = 0; k < 6; ++k) ep[CBEV_E_ABS_ACCEL_LONG + k] = (sa[S_C0 + k] + cm6[k]) / ep_len;
          ep[CBEV_E_VIOL_RATE] = ep_viol / ep_len; ep[CBEV_E_HARSH_RATE] = ep_harsh / ep_len;
          ep[CBEV_E_SCENE] = (double)scene; ep[CBEV_E_NUM_VEHICLES] = (double)pool.num_vehicles[scene];
          ep[CBEV_E_LEN_ROUTE] = pool.len_ego_route[scene]; ep[CBEV_E_EPISODE] = (double)st.episode[env];
        }
        atomicAdd(gstats + CBEV_S_EPISODES, 1.0);
        atomicAdd(gstats + CBEV_S_RETURN, ep_ret);
        atomicAdd(gstats + CBEV_S_LENGTH, ep_len);
        atomicAdd(gstats + CBEV_S_MEAN_SPEED, ep_speed * inv);
        atomicAdd(gstats + CBEV_S_CAUSE0 + (int)ep_cause, 1.0);
        for (int k = 0; k < 6; ++k) atomicAdd(gstats + CBEV_S_ABS_COMFORT0 + k, (sa[S_C0 + k] + cm6[k]) * inv);
        atomicAdd(gstats + CBEV_S_VIOL_RATE, ep_viol * inv);
        atomicAdd(gstats + CBEV_S_HARSH_RATE, ep_harsh * inv);
        st.episode[env] += 1;
        st.done[env] = 1;
        if constexpr (MODE == JG_LIVE)
          move_order[atomicAdd(move_cnt, 1)] = env;  // resets next step: grouped at the front of k_move's env order
        for (int k = 0; k < S_SLOTS; ++k) sa[k] = 0.0;  // stats.reset() after terminated(), stats.py:107-112
      } else {
        if constexpr (MODE == JG_LIVE) move_order[P.N - 1 - atomicAdd(move_cnt + 1, 1)] = env;
        sa[S_RET] = ep_ret; sa[S_LEN] = ep_len; sa[S_SPEED] = ep_speed;
        for (int k = 0; k < 6; ++k) sa[S_C0 + k] += cm6[k];
        sa[S_VIOL] = ep_viol; sa[S_HARSH] = ep_harsh; sa[S_CAUSE] = ep_cause;
      }
    }
    if (hero_now) {
      double* hb = hb_s;
      hb[CBEV_H_X] = e.x; hb[CBEV_H_Y] = e.y; hb[CBEV_H_YAW] = e.yaw; hb[CBEV_H_V] = e.v;
      hb[CBEV_H_X1] = e.x1; hb[CBEV_H_Y1] = e.y1; hb[CBEV_H_YAW1] = e.yaw1; hb[CBEV_H_V1] = e.v1;
      hb[CBEV_H_DIST2WP] = dist2wp; hb[CBEV_H_SP_X] = ecx[tidx]; hb[CBEV_H_SP_Y] = ecy[tidx];
      hb[CBEV_H_SP_YAW] = ecyaw[tidx];
      hb[CBEV_H_CMD_GAS] = eg[E_GAS]; hb[CBEV_H_CMD_STEER] = eg[E_STEER]; hb[CBEV_H_CMD_BRAKE] = eg[E_BRAKE];
      hb[CBEV_H_DELTA] = eg[E_DELTA];
      hb[CBEV_H_SPEED_MPS] = speed_mps; hb[CBEV_H_ACCEL_LONG] = accel_long; hb[CBEV_H_ACCEL_LAT] = accel_lat;
      hb[CBEV_H_JERK_LONG] = jerk_long; hb[CBEV_H_JERK_LAT] = jerk_lat; hb[CBEV_H_YAW_RATE] = yaw_rate_deg;
      hb[CBEV_H_YAW_ACC] = yaw_acc;
      hb[CBEV_H_ACC] = acc; hb[CBEV_H_TIDX] = (double)tidx; hb[CBEV_H_HIT] = (double)hit;
      hb[CBEV_H_HIT_ID] = (double)hit_id; hb[CBEV_H_TILE] = (double)tile; hb[CBEV_H_NEARBY] = (double)n_nearby;
      hb[CBEV_H_DIST2GOAL] = d2g; hb[CBEV_H_T] = t_sim; hb[CBEV_H_SCENE] = (double)scene;
    }
  }
  __syncwarp(GM);
  if (hero_now) {
    for (int f = lane; f < CBEV_HERO_FIELDS; f += G) out.hero[(size_t)env * CBEV_HERO_FIELDS + f] = hb_s[f];
  }
  reward_out = reward;
  terminated_out = terminated;
  truncated_out = truncated;
  cause_out = cause;
}

template <int G>
__global__ void __launch_bounds__(32 * CBEV_WARPS_PER_BLOCK, 4)
k_judge(SimParams P, PoolDev pool, EnvState st, cbev_step_out out, const int32_t* __restrict__ desc,
        double* __restrict__ gstats, int32_t* __restrict__ move_order, int32_t* __restrict__ move_cnt) {
  constexpr int EPW = 32 / G;  // environments per warp
  __shared__ double s_hero[CBEV_WARPS_PER_BLOCK][EPW][CBEV_HERO_FIELDS];
  const Group<G> g(P);
  const int lane = g.lane, env = g.env;
  if (env >= P.N) return;
  if (desc[(size_t)env * CBEV_DESC_WORDS + RD_FLAGS] & 1) {  // auto-reset this step: k_move wrote the outputs
    if (lane == 0) move_order[P.N - 1 - atomicAdd(move_cnt + 1, 1)] = env;
    return;
  }
  double reward;
  bool terminated, truncated;
  int cause;
  judge_body<G, JG_LIVE>(P, pool, st, out, gstats, move_order, move_cnt, s_hero[g.warp][g.grp], env, lane, g.gb, g.GM,
                       false, reward, terminated, truncated, cause);
}

// Action repeat (cbev_set_action_repeat): one group of G lanes per env runs up to `repeat` simulator steps with the
// same action, move_body + judge_body back to back as in k_lookahead, on the live state.  An env whose last agent step
// was terminal (NEXT_STEP) auto-resets instead, exactly as in k_move.  Every other env stops after its first terminal
// sub-step; its descriptor and draw list are those of its last sub-step (MV_BRANCH_DRAW: the live step's drawing
// without auto-reset and CTA order, so each sub-step draws -- which one is last is known only after its judge), and
// the raster launch after this kernel renders that one frame.  The outputs are those of the last sub-step, except the
// reward: the sub-step rewards summed in order, unfused, from the first (so repeat = 1 returns it bit for bit).
// move_order is this launch's env permutation, so nothing here writes it (a late block would read entries an earlier
// one overwrote): it stays the permutation the last k_judge / k_reset left, and order only affects speed.
template <int G>
__global__ void __launch_bounds__(32 * CBEV_WARPS_PER_BLOCK, 4)
k_step_repeat(SimParams P, PoolDev pool, EnvState st, const void* __restrict__ actions, cbev_step_out out,
              int32_t* __restrict__ desc, uint32_t* __restrict__ rects, int32_t* __restrict__ order,
              int32_t* __restrict__ order_cnt, double* __restrict__ gstats, const int32_t* __restrict__ move_order,
              int32_t repeat) {
  constexpr int EPW = 32 / G;
  __shared__ double s_hero[CBEV_WARPS_PER_BLOCK][EPW][CBEV_HERO_FIELDS];
  const Group<G> g(P, move_order);
  const int lane = g.lane, env = g.env;
  if (env >= P.N) return;
  if (P.autoreset == CBEV_AUTORESET_NEXT_STEP && st.done[env]) {
    auto_reset_env<G>(P, pool, st, out, desc + (size_t)env * CBEV_DESC_WORDS, order, order_cnt, env, lane, g.GM);
    return;
  }
  double sum = 0.0;
  for (int k = 0; k < repeat; ++k) {
    move_body<G, MV_BRANCH_DRAW>(P, pool, st, actions, out, desc, rects, nullptr, nullptr, env, lane, g.gb, g.GM);
    __syncwarp(g.GM);  // lane 0 stored the new ego pose; every lane of the group reads it
    double r;
    bool terminated, truncated;
    int cause;
    judge_body<G, JG_LIVE_REPEAT>(P, pool, st, out, gstats, nullptr, nullptr, s_hero[g.warp][g.grp], env, lane, g.gb,
                                  g.GM, k == repeat - 1, r, terminated, truncated, cause);
    sum = k == 0 ? r : __dadd_rn(sum, r);
    if (terminated || truncated) break;  // uniform across the group
  }
  if (lane == 0) {
    out.reward[env] = sum;
    order[P.N - 1 - atomicAdd(order_cnt + 1, 1)] = env;  // light: one frame
  }
}

// Same-step auto-reset (CBEV_AUTORESET_SAME_STEP), after the step's raster kernel: CTA b resets env b if its call
// ended (terminated or truncated; judge_body sets done exactly then) -- the NEXT_STEP scene draw, reset_env, the reset
// descriptor header and a place at the front of the raster order -- and gives every other env the skip header and a
// place at the back.  The terminal windows are copied in `slices` byte ranges of the F-frame window, slice j of env e
// by CTA (e + j) mod N, so one finished env's copy is spread over that many SMs instead of forming a one-SM tail.  The
// ended flags of the (up to 32) envs a CTA serves are read once, in parallel, into a bit mask: bit j = env (b - j).
// Neither the step outputs nor move_order (k_judge's order for the next k_move) are written, nor the ring: the raster
// launch at the same head that follows renders the reset frames into every window slot.
#define CBEV_SSR_THREADS 256
struct SameStepArgs {
  const uint8_t* terminated;
  const uint8_t* truncated;
  int32_t* desc;
  int32_t* order;
  int32_t* order_cnt;
  const uint8_t* ring;  // window of env e: ring + e * ring_row + win_off, win bytes
  uint8_t* final_obs;   // [N][win] or null
  int64_t ring_row, win_off, win, slice;
  int32_t slices;       // 1..32
};

__global__ void __launch_bounds__(CBEV_SSR_THREADS)
k_same_step_reset(SimParams P, PoolDev pool, EnvState st, const SameStepArgs a) {
  __shared__ unsigned s_ended;
  const int b = blockIdx.x, tid = threadIdx.x, N = P.N;
  if (tid < 32) {
    bool ended = false;
    if (tid < a.slices) {
      const int env = ((b - tid) % N + N) % N;
      ended = (a.terminated[env] | a.truncated[env]) != 0;
    }
    const unsigned m = __ballot_sync(0xffffffffu, ended);
    if (tid == 0) s_ended = m;
  }
  __syncthreads();
  const unsigned ended = s_ended;
  if (a.final_obs != nullptr) {
    for (int j = 0; j < a.slices; ++j) {
      if (!((ended >> j) & 1u)) continue;
      const int env = ((b - j) % N + N) % N;
      const int64_t lo = (int64_t)j * a.slice, hi = min(lo + a.slice, a.win);
      const uint4* src = (const uint4*)(a.ring + (size_t)env * a.ring_row + a.win_off + lo);
      uint4* dst = (uint4*)(a.final_obs + (size_t)env * a.win + lo);
      const int n = (int)((hi - lo) >> 4);
      int i = tid;
      for (; i + 3 * CBEV_SSR_THREADS < n; i += 4 * CBEV_SSR_THREADS) {  // four 16-byte loads in flight per thread
        const uint4 v0 = __ldg(src + i), v1 = __ldg(src + i + CBEV_SSR_THREADS);
        const uint4 v2 = __ldg(src + i + 2 * CBEV_SSR_THREADS), v3 = __ldg(src + i + 3 * CBEV_SSR_THREADS);
        dst[i] = v0; dst[i + CBEV_SSR_THREADS] = v1; dst[i + 2 * CBEV_SSR_THREADS] = v2; dst[i + 3 * CBEV_SSR_THREADS] = v3;
      }
      for (; i < n; i += CBEV_SSR_THREADS) dst[i] = __ldg(src + i);
    }
  }
  if (tid >= 32) return;
  const int env = b, lane = tid;
  int32_t* d = a.desc + (size_t)env * CBEV_DESC_WORDS;
  if (!(ended & 1u)) {
    if (lane == 0) {
      d[RD_FLAGS] = 2;  // bit1: the raster launch skips this env
      a.order[N - 1 - atomicAdd(a.order_cnt + 1, 1)] = env;
    }
    return;
  }
  const int scene = auto_reset_scene(P, pool, st, env);  // episode was advanced by the terminal step's judging
  __syncwarp();
  reset_env(P, pool, st, env, scene, lane);
  if (lane == 0) {
    a.order[atomicAdd(a.order_cnt, 1)] = env;  // the reset frames go first: F window slots each
    const double* s0 = pool.ego_state0 + (size_t)scene * 4;
    View v;
    compute_view(P, s0[0], s0[1], 0.0, v);
    write_desc_header(P, d, v, 0, 1, crop_corner_class(P, v));  // bit0: reset frame
  }
}

// Roll every scene's scripted actors out for traj_steps steps (one warp per scene) and record the poses.
__global__ void __launch_bounds__(32 * CBEV_WARPS_PER_BLOCK)
k_rollout(SimParams P, PoolDev pool) {
  const int scene = blockIdx.x * CBEV_WARPS_PER_BLOCK + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (scene >= pool.n_scenes) return;
  const int A0 = pool.actor_off[scene], A = pool.actor_off[scene + 1] - A0;
  init_actors(P, pool, pool.roll, (size_t)scene, scene, lane, 32);
  __syncwarp();
  double t_sim = 0.0;
  for (int step = 0; step < pool.traj_steps; ++step) {
    t_sim += DT;  // scene.py:91
    for (int base = 0; base < A; base += 32) {
      const int a = base + lane;
      const bool has = a < A;
      const int ga = A0 + (has ? a : 0);
      const size_t o = (size_t)scene * P.max_actors + (has ? a : 0);
      Body b;
      int kind = 0;
      actor_chunk_step<32>(P, pool, pool.roll, (size_t)scene, ga, o, has, t_sim, lane, 0, FULL, b, kind);
      if (has) pool.traj[pool.traj_off[scene] + (size_t)step * A + a] = make_double4(b.x, b.y, b.yaw, b.v);
    }
    __syncwarp();
  }
}

struct LookaheadArgs {
  const uint8_t* src[CBEV_STATE_SECTIONS];  // live state sections (env rows)
  uint8_t* dst[CBEV_STATE_SECTIONS];        // branch state sections (branch rows), same per-env counts
  int32_t esize[CBEV_STATE_SECTIONS], count[CBEV_STATE_SECTIONS];
  const int32_t* live_scene;
  const uint8_t* live_done;
  const int32_t* roots;  // [B] or null = identity
  const void* actions;   // [H][B] int64 or [H][B][3] float32
  double gamma;
  int32_t n_live, horizon;
  cbev_lookahead_out out;
};

// Draw records of k_lookahead_obs (engine-owned, api.cu: ensure_branch_render).  Step t of branch b records its
// descriptor and draw list in staging slot t mod F; the epilogue copies the last min(steps, F) of them to render
// position b * F + f (window position f, oldest first), where the raster kernel, which uses one index for the
// descriptor and the output frame, renders them into the caller's [B][F] windows.
struct LookaheadRender {
  int32_t* stage_desc;    // [F][B][CBEV_DESC_WORDS]
  uint32_t* stage_rects;  // [F][B][max_rects][CBEV_RECT_WORDS]
  int32_t* desc;          // [B * F][CBEV_DESC_WORDS]
  uint32_t* rects;        // [B * F][max_rects][CBEV_RECT_WORDS]
  int32_t F;
};

// Roots of cbev_lookahead_ex beyond what LookaheadArgs carries.  ROWS: branch b starts from row roots[b] of a
// snapshot (layout SnapLayout at the rows' retreat slots) instead of a live env; the scene and the done flag come from
// the row header, and a row taken at fewer retreat slots leaves the slots it lacks zeroed, as k_restore does.  LEAF:
// the header of a live root (its episode counter) for the leaf rows.
struct LookaheadRoots {
  const int32_t* live_episode;
  const uint8_t* rows;
  int64_t row_bytes;
  int64_t off[CBEV_STATE_SECTIONS];    // row offset of each state section
  int32_t count[CBEV_STATE_SECTIONS];  // elements per row (row side)
  int32_t n_rows;
};

// One group of G lanes per branch (P.N = number of branches) runs all H steps: the root's state is copied into the
// branch row, then each step is move_body + judge_body of the branch instantiation, back to back.  Branches are
// independent, so the whole call is one launch without grid-wide synchronisation.  OBS: every step also records its
// draw list (MV_BRANCH_DRAW), and the epilogue lays out the render positions of the branch's leaf window.  ROWS: the
// roots are snapshot rows (LookaheadRoots).  LEAF: the branch row becomes a snapshot row afterwards (k_leaf_rows), so
// it also keeps the header (scene, episode, done) and the episode accumulators (JG_BRANCH_ROW); every valid root is
// copied, terminal ones included (their leaf row is the root's own), and an invalid one gets scene = -1 (no row).
// REPEAT: step t is an agent step of up to `repeat` sub-steps with action row t, k_step_repeat's loop: it stops at
// the first terminal sub-step, sums the sub-step rewards in order, and every sub-step draws into staging slot t, so
// the slot holds the record of the last one.
template <int G, bool OBS, bool ROWS = false, bool LEAF = false, bool REPEAT = false>
__device__ __forceinline__ void lookahead_body(const SimParams& P, const PoolDev& pool, const EnvState& br,
                                               const LookaheadArgs& a, const LookaheadRender& rd,
                                               const LookaheadRoots& rr = LookaheadRoots{}, int32_t repeat = 1) {
  constexpr int EPW = 32 / G;
  __shared__ double s_hero[CBEV_WARPS_PER_BLOCK][EPW][CBEV_HERO_FIELDS];
  const Group<G> g(P);
  const int lane = g.lane, b = g.env, B = P.N, H = a.horizon;
  const unsigned GM = g.GM;
  if (b >= B) return;
  const int root = a.roots ? a.roots[b] : b;
  bool live, valid;
  int4 hdr = make_int4(-1, 0, 1, 0);  // ROWS: the root row's header (scene, episode, done)
  const uint8_t* row = nullptr;
  if constexpr (ROWS) {
    // device roots are trusted, never used OOB; nor is a header scene outside the pool
    valid = root >= 0 && root < rr.n_rows;
    if (valid) {
      row = rr.rows + (size_t)root * rr.row_bytes;
      hdr = *(const int4*)row;
    }
    valid = valid && hdr.x >= 0 && hdr.x < pool.n_scenes;
    live = valid && (uint8_t)hdr.z == 0;
  } else if constexpr (LEAF) {
    valid = root >= 0 && root < a.n_live;
    live = valid && a.live_done[root] == 0;
  } else {
    live = root >= 0 && root < a.n_live && a.live_done[root] == 0;  // device roots are trusted, never used OOB
    valid = live;
  }
  if (LEAF ? valid : live) {
    if (lane == 0) {
      if constexpr (ROWS) br.scene[b] = hdr.x;
      else br.scene[b] = a.live_scene[root];
      if constexpr (LEAF) {
        br.episode[b] = ROWS ? hdr.y : rr.live_episode[root];
        br.done[b] = ROWS ? (uint8_t)hdr.z : a.live_done[root];
      }
    }
#pragma unroll 1
    for (int s = 0; s < CBEV_STATE_SECTIONS; ++s) {
      const int es = a.esize[s], n = a.count[s];
      uint8_t* dp = a.dst[s] + (size_t)b * n * es;
      if constexpr (ROWS) {
        const int nr = rr.count[s];
        const uint8_t* sp = row + rr.off[s];
        for (int i = lane; i < n; i += G) {
          if (i < nr) cbev_copy_elem(dp + (size_t)i * es, sp + (size_t)i * es, es);
          else cbev_zero_elem(dp + (size_t)i * es, es);
        }
      } else {
        const uint8_t* sp = a.src[s] + (size_t)root * n * es;
        for (int i = lane; i < n; i += G) cbev_copy_elem(dp + (size_t)i * es, sp + (size_t)i * es, es);
      }
    }
  }
  if constexpr (LEAF) {
    if (!valid && lane == 0) br.scene[b] = -1;
  }
  __syncwarp(GM);
  const cbev_lookahead_out& o = a.out;
  cbev_step_out so = {};
  so.hero = o.hero;
  double ret = 0.0, w = 1.0;
  int steps = 0, cause = CBEV_CAUSE_NONE;
  bool terminated = false, truncated = false;
  if (live) {
    int slot = 0;  // OBS: t mod F
    for (int t = 0; t < H; ++t) {
      const void* act = P.action_mode == CBEV_ACTION_DISCRETE
                            ? (const void*)((const long long*)a.actions + (size_t)t * B)
                            : (const void*)((const float*)a.actions + (size_t)t * B * 3);
      double r;
      if constexpr (REPEAT) {
        for (int k = 0; k < repeat; ++k) {  // the sub-steps of agent step t, as in k_step_repeat
          if constexpr (OBS) {
            move_body<G, MV_BRANCH_DRAW>(P, pool, br, act, so, rd.stage_desc + (size_t)slot * B * CBEV_DESC_WORDS,
                                         rd.stage_rects + (size_t)slot * B * P.max_rects * CBEV_RECT_WORDS, nullptr,
                                         nullptr, b, lane, g.gb, GM);
          } else {
            move_body<G, MV_BRANCH>(P, pool, br, act, so, nullptr, nullptr, nullptr, nullptr, b, lane, g.gb, GM);
          }
          __syncwarp(GM);  // lane 0 stored the new ego pose; every lane of the group reads it
          double rk;
          judge_body<G, LEAF ? JG_BRANCH_ROW : JG_BRANCH>(P, pool, br, so, nullptr, nullptr, nullptr,
                                                          s_hero[g.warp][g.grp], b, lane, g.gb, GM,
                                                          t == H - 1 && k == repeat - 1, rk, terminated, truncated,
                                                          cause);
          r = k == 0 ? rk : __dadd_rn(r, rk);  // in sub-step order, unfused: j = 1 gives r1 bit for bit
          if (terminated || truncated) break;  // uniform across the group
        }
        if constexpr (OBS) slot = slot + 1 == rd.F ? 0 : slot + 1;  // slot t holds the last sub-step's record
      } else {
        if constexpr (OBS) {
          move_body<G, MV_BRANCH_DRAW>(P, pool, br, act, so, rd.stage_desc + (size_t)slot * B * CBEV_DESC_WORDS,
                                       rd.stage_rects + (size_t)slot * B * P.max_rects * CBEV_RECT_WORDS, nullptr,
                                       nullptr, b, lane, g.gb, GM);
          slot = slot + 1 == rd.F ? 0 : slot + 1;
        } else {
          move_body<G, MV_BRANCH>(P, pool, br, act, so, nullptr, nullptr, nullptr, nullptr, b, lane, g.gb, GM);
        }
        __syncwarp(GM);  // lane 0 stored the new ego pose; every lane of the group reads it
        judge_body<G, LEAF ? JG_BRANCH_ROW : JG_BRANCH>(P, pool, br, so, nullptr, nullptr, nullptr,
                                                        s_hero[g.warp][g.grp], b, lane, g.gb, GM, t == H - 1, r,
                                                        terminated, truncated, cause);
      }
      if (lane == 0 && o.reward) o.reward[(size_t)t * B + b] = r;
      ret = __dadd_rn(ret, __dmul_rn(w, r));  // unfused, in step order: reproducible from reward[]
      w = __dmul_rn(w, a.gamma);
      steps = t + 1;
      if (terminated || truncated) break;  // uniform across the group
    }
  }
  if (o.reward)
    for (int t = steps + lane; t < H; t += G) o.reward[(size_t)t * B + b] = 0.0;
  if (steps == 0 && o.hero)
    for (int f = lane; f < CBEV_HERO_FIELDS; f += G) o.hero[(size_t)b * CBEV_HERO_FIELDS + f] = 0.0;
  if (lane == 0) {
    o.ret[b] = ret;
    if (o.steps) o.steps[b] = steps;
    if (o.terminated) o.terminated[b] = terminated;
    if (o.truncated) o.truncated[b] = truncated;
    if (o.cause) o.cause[b] = (uint8_t)cause;
  }
  if constexpr (OBS) {
    // Every render position of the branch is written on every call: window position f < F - min(steps, F) belongs to
    // the root's window (k_leaf_window) and gets a skip header, the others the record of step steps - F + f.
    __syncwarp(GM);  // the records of the last step were written by other lanes of the group
    const int F = rd.F, first = F - (steps < F ? steps : F);
    const int RW = P.max_rects * CBEV_RECT_WORDS;
    for (int f = 0; f < F; ++f) {
      int32_t* dd = rd.desc + ((size_t)b * F + f) * CBEV_DESC_WORDS;
      if (f < first) {
        if (lane == 0) dd[RD_FLAGS] = 2;  // bit1: the raster kernel skips this position
        continue;
      }
      const int j = (steps - F + f) % F;
      const int32_t* sd = rd.stage_desc + ((size_t)j * B + b) * CBEV_DESC_WORDS;
      for (int k = lane; k < CBEV_DESC_WORDS; k += G) dd[k] = sd[k];
      const int nw = sd[RD_NRECTS] * CBEV_RECT_WORDS;
      const uint32_t* sr = rd.stage_rects + ((size_t)j * B + b) * RW;
      uint32_t* dr = rd.rects + ((size_t)b * F + f) * RW;
      for (int k = lane; k < nw; k += G) dr[k] = sr[k];
    }
  }
}

template <int G>
__global__ void __launch_bounds__(32 * CBEV_WARPS_PER_BLOCK, 4)
k_lookahead(SimParams P, PoolDev pool, EnvState br, LookaheadArgs a) {
  lookahead_body<G, false>(P, pool, br, a, LookaheadRender{});
}

template <int G>
__global__ void __launch_bounds__(32 * CBEV_WARPS_PER_BLOCK, 4)
k_lookahead_obs(SimParams P, PoolDev pool, EnvState br, LookaheadArgs a, LookaheadRender rd) {
  lookahead_body<G, true>(P, pool, br, a, rd);
}

// cbev_lookahead_ex beyond the two kernels above: roots from snapshot rows (ROWS) and / or leaf rows (LEAF, which
// needs the draw records: OBS)
template <int G, bool OBS, bool ROWS, bool LEAF>
__global__ void __launch_bounds__(32 * CBEV_WARPS_PER_BLOCK, 4)
k_lookahead_ex(SimParams P, PoolDev pool, EnvState br, LookaheadArgs a, LookaheadRender rd, LookaheadRoots rr) {
  lookahead_body<G, OBS, ROWS, LEAF>(P, pool, br, a, rd, rr);
}

// cbev_lookahead_repeat: the modes of the kernels above with agent steps of up to `repeat` > 1 sub-steps each (REPEAT)
template <int G, bool OBS, bool ROWS, bool LEAF>
__global__ void __launch_bounds__(32 * CBEV_WARPS_PER_BLOCK, 4)
k_lookahead_rep(SimParams P, PoolDev pool, EnvState br, LookaheadArgs a, LookaheadRender rd, LookaheadRoots rr,
                int32_t repeat) {
  lookahead_body<G, OBS, ROWS, LEAF, true>(P, pool, br, a, rd, rr, repeat);
}

}  // namespace

static SimParams make_params(cbev_engine* e) {
  SimParams P;
  P.N = e->N;
  P.max_actors = e->cfg.max_actors;
  P.max_rects = e->max_rects;
  P.max_retreat = e->pool.max_retreat;
  P.map_w = e->map_w;
  P.map_h = e->map_h;
  P.fov = e->cfg.fov_size;
  P.hero_scale = (float)(1024 / e->cfg.fov_size);  // hero.py:14
  P.hero_w = 32 / (1024 / e->cfg.fov_size);        // hero.py:17
  P.win_max = e->win_max;
  P.crop = e->crop;
  P.pad = e->pad;
  P.anchor_x = e->anchor_x;
  P.anchor_y = e->anchor_y;
  P.action_mode = e->cfg.action_mode;
  P.n_discrete = e->cfg.n_discrete;
  P.reward_mode = e->cfg.reward_mode;
  // SAME_STEP resets an env in its terminal call (k_same_step_reset); an env that starts a call done (a restored
  // terminal row) auto-resets in k_move / k_step_repeat exactly as under NEXT_STEP
  P.autoreset = e->cfg.autoreset == CBEV_AUTORESET_SAME_STEP ? CBEV_AUTORESET_NEXT_STEP : e->cfg.autoreset;
  P.seed = e->cfg.seed;
  P.map = e->map;
  for (int i = 0; i < 48; ++i) P.discrete_table[i] = e->cfg.discrete_table[i];
  P.cfg = e->cfg;
  return P;
}

void cbev_launch_reset(cbev_engine* e, const uint8_t* mask, const int32_t* scene_ids, cudaStream_t s) {
  SimParams P = make_params(e);
  int blocks = (e->N + CBEV_WARPS_PER_BLOCK - 1) / CBEV_WARPS_PER_BLOCK;
  k_reset<<<blocks, 32 * CBEV_WARPS_PER_BLOCK, 0, s>>>(P, e->pool, e->st, mask, scene_ids, e->desc, e->order, e->move_order);
  e->launches += 1;
}

static bool narrow_groups(const cbev_engine* e) {
  return e->pool.max_actors <= 8 || e->pool.traj_steps > 0;  // table look-ups need no wide actor loops
}

void cbev_launch_move(cbev_engine* e, const void* actions, const cbev_step_out* out, cudaStream_t s) {
  SimParams P = make_params(e);
  const int32_t* mo = (e->debug_flags & CBEV_DBG_IDENTITY_MOVE_ORDER) ? nullptr : e->move_order;
  if (narrow_groups(e)) {
    constexpr int G = 8;
    int per_block = CBEV_WARPS_PER_BLOCK * (32 / G);
    int blocks = (e->N + per_block - 1) / per_block;
    k_move<G><<<blocks, 32 * CBEV_WARPS_PER_BLOCK, 0, s>>>(P, e->pool, e->st, actions, *out, e->desc, e->rects, e->order,
                                                           e->order_cnt, mo, e->move_cnt);
  } else {
    int blocks = (e->N + CBEV_WARPS_PER_BLOCK - 1) / CBEV_WARPS_PER_BLOCK;
    k_move<32><<<blocks, 32 * CBEV_WARPS_PER_BLOCK, 0, s>>>(P, e->pool, e->st, actions, *out, e->desc, e->rects, e->order,
                                                            e->order_cnt, mo, e->move_cnt);
  }
  e->launches += 1;
}

void cbev_launch_judge(cbev_engine* e, const cbev_step_out* out, cudaStream_t s) {
  SimParams P = make_params(e);
  // the judging loops over actors / route segments are cheap per element: 8 lanes per env unless routes are long
  constexpr int G = 8;
  int per_block = CBEV_WARPS_PER_BLOCK * (32 / G);
  int blocks = (e->N + per_block - 1) / per_block;
  k_judge<G><<<blocks, 32 * CBEV_WARPS_PER_BLOCK, 0, s>>>(P, e->pool, e->st, *out, e->desc, e->gstats, e->move_order,
                                                          e->move_cnt);
  e->launches += 1;
}

void cbev_launch_step_repeat(cbev_engine* e, const void* actions, const cbev_step_out* out, cudaStream_t s) {
  SimParams P = make_params(e);
  const int32_t* mo = (e->debug_flags & CBEV_DBG_IDENTITY_MOVE_ORDER) ? nullptr : e->move_order;
  constexpr int T = 32 * CBEV_WARPS_PER_BLOCK;
  // group width as in k_move
  if (narrow_groups(e)) {
    constexpr int G = 8;
    const int blocks = (e->N + CBEV_WARPS_PER_BLOCK * (32 / G) - 1) / (CBEV_WARPS_PER_BLOCK * (32 / G));
    k_step_repeat<G><<<blocks, T, 0, s>>>(P, e->pool, e->st, actions, *out, e->desc, e->rects, e->order, e->order_cnt,
                                          e->gstats, mo, e->action_repeat);
  } else {
    const int blocks = (e->N + CBEV_WARPS_PER_BLOCK - 1) / CBEV_WARPS_PER_BLOCK;
    k_step_repeat<32><<<blocks, T, 0, s>>>(P, e->pool, e->st, actions, *out, e->desc, e->rects, e->order, e->order_cnt,
                                           e->gstats, mo, e->action_repeat);
  }
  e->launches += 1;
}

void cbev_launch_same_step_reset(cbev_engine* e, const cbev_step_out* out, int32_t head, cudaStream_t s) {
  SimParams P = make_params(e);
  const int F = e->cfg.frame_stack;
  SameStepArgs a;
  a.terminated = out->terminated;
  a.truncated = out->truncated;
  a.desc = e->desc;
  a.order = e->order;
  a.order_cnt = e->order_cnt;
  a.ring = (const uint8_t*)e->ring;
  a.final_obs = (uint8_t*)e->final_obs;
  a.ring_row = (int64_t)e->cfg.ring_slots * e->frame_bytes;
  a.win_off = (int64_t)(head - F + 1) * e->frame_bytes;
  a.win = (int64_t)F * e->frame_bytes;
  // slices of >= 16 KB (at most 32, the CTAs that share one window copy), 16-byte multiples
  const int64_t min_slice = 16 << 10;
  int64_t slices = (a.win + min_slice - 1) / min_slice;
  if (slices > 32) slices = 32;
  a.slice = ((a.win + slices - 1) / slices + 15) & ~(int64_t)15;
  a.slices = (int32_t)((a.win + a.slice - 1) / a.slice);
  k_same_step_reset<<<e->N, CBEV_SSR_THREADS, 0, s>>>(P, e->pool, e->st, a);
  e->launches += 1;
}

// One lookahead mode: repeat 1 runs the kernel of cbev_lookahead / _obs / _ex, a larger repeat its k_lookahead_rep.
template <int G, bool OBS, bool ROWS, bool LEAF>
static void launch_lookahead_mode(int blocks, cudaStream_t s, int32_t repeat, const SimParams& P, cbev_engine* e,
                                  const LookaheadArgs& a, const LookaheadRender& rd, const LookaheadRoots& rr) {
  constexpr int T = 32 * CBEV_WARPS_PER_BLOCK;
  if (repeat > 1) {
    k_lookahead_rep<G, OBS, ROWS, LEAF><<<blocks, T, 0, s>>>(P, e->pool, e->branch, a, rd, rr, repeat);
  } else if constexpr (!ROWS && !LEAF) {
    if constexpr (OBS) k_lookahead_obs<G><<<blocks, T, 0, s>>>(P, e->pool, e->branch, a, rd);
    else k_lookahead<G><<<blocks, T, 0, s>>>(P, e->pool, e->branch, a);
  } else {
    k_lookahead_ex<G, OBS, ROWS, LEAF><<<blocks, T, 0, s>>>(P, e->pool, e->branch, a, rd, rr);
  }
}

template <int G>
static void launch_lookahead(int blocks, cudaStream_t s, bool record, bool rows, bool leaf, int32_t repeat,
                             const SimParams& P, cbev_engine* e, const LookaheadArgs& a, const LookaheadRender& rd,
                             const LookaheadRoots& rr) {
  if (leaf) {  // leaf rows carry frames: always recorded
    if (rows) launch_lookahead_mode<G, true, true, true>(blocks, s, repeat, P, e, a, rd, rr);
    else launch_lookahead_mode<G, true, false, true>(blocks, s, repeat, P, e, a, rd, rr);
  } else if (rows) {
    if (record) launch_lookahead_mode<G, true, true, false>(blocks, s, repeat, P, e, a, rd, rr);
    else launch_lookahead_mode<G, false, true, false>(blocks, s, repeat, P, e, a, rd, rr);
  } else {
    if (record) launch_lookahead_mode<G, true, false, false>(blocks, s, repeat, P, e, a, rd, rr);
    else launch_lookahead_mode<G, false, false, false>(blocks, s, repeat, P, e, a, rd, rr);
  }
}

void cbev_launch_lookahead(cbev_engine* e, const int32_t* roots, int32_t n_branches, int32_t horizon,
                           const void* actions, double gamma, const cbev_lookahead_out* out, bool record,
                           const RowSource* rows, bool leaf, int32_t repeat, cudaStream_t s) {
  SimParams P = make_params(e);
  P.N = n_branches;
  LookaheadArgs a;
  const int32_t A = e->cfg.max_actors > 0 ? e->cfg.max_actors : 1, R = e->pool.max_retreat;
  const StateSections src = cbev_state_sections(e->st, A, R), dst = cbev_state_sections(e->branch, A, R);
  for (int k = 0; k < CBEV_STATE_SECTIONS; ++k) {
    a.src[k] = (const uint8_t*)*src.field[k];
    a.dst[k] = (uint8_t*)*dst.field[k];
    a.esize[k] = src.esize[k];
    a.count[k] = src.count[k];
  }
  a.live_scene = e->st.scene;
  a.live_done = e->st.done;
  a.roots = roots;
  a.actions = actions;
  a.gamma = gamma;
  a.n_live = e->N;
  a.horizon = horizon;
  a.out = *out;
  // record: the draw records of the leaf windows (cbev_lookahead_obs), into the branch render state
  const LookaheadRender rd{e->br_stage_desc, e->br_stage_rects, e->br_desc, e->br_rects, e->cfg.frame_stack};
  LookaheadRoots rr = {};
  rr.live_episode = e->st.episode;
  if (rows) {
    rr.rows = (const uint8_t*)rows->rows;
    rr.row_bytes = rows->L.row_bytes;
    for (int k = 0; k < CBEV_STATE_SECTIONS; ++k) {
      rr.off[k] = rows->L.off[k];
      rr.count[k] = rows->L.count[k];
    }
    rr.n_rows = rows->n_rows;
  }
  // group width as in k_move: the branch steps its actors the way the live step does
  if (narrow_groups(e)) {
    constexpr int G = 8;
    const int blocks = (n_branches + CBEV_WARPS_PER_BLOCK * (32 / G) - 1) / (CBEV_WARPS_PER_BLOCK * (32 / G));
    launch_lookahead<G>(blocks, s, record, rows != nullptr, leaf, repeat, P, e, a, rd, rr);
  } else {
    const int blocks = (n_branches + CBEV_WARPS_PER_BLOCK - 1) / CBEV_WARPS_PER_BLOCK;
    launch_lookahead<32>(blocks, s, record, rows != nullptr, leaf, repeat, P, e, a, rd, rr);
  }
  e->launches += 1;
}

void cbev_launch_rollout(cbev_engine* e, cudaStream_t s) {
  SimParams P = make_params(e);
  int blocks = (e->pool.n_scenes + CBEV_WARPS_PER_BLOCK - 1) / CBEV_WARPS_PER_BLOCK;
  k_rollout<<<blocks, 32 * CBEV_WARPS_PER_BLOCK, 0, s>>>(P, e->pool);
  e->launches += 1;
}

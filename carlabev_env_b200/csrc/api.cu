// api.cu -- the C ABI of include/cbev.h: engine lifetime, uploads, reset / step orchestration.
#include <cuda.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <new>
#include <random>
#include <vector>

#include "engine.h"

static thread_local char g_err[512] = "";

void cbev_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

#define CU_TRY(expr)                                                                       \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      cbev_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return CBEV_ERR_CUDA;                                                                \
    }                                                                                      \
  } while (0)

namespace {

// CBEV_DEBUG_SYNC=1: synchronise after every kernel and report which one faulted
int debug_sync(const char* what, cudaStream_t s) {
  static const bool on = getenv("CBEV_DEBUG_SYNC") != nullptr;
  if (!on) return CBEV_OK;
  cudaError_t e = cudaStreamSynchronize(s);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) {
    cbev_set_error("kernel %s failed: %s", what, cudaGetErrorString(e));
    return CBEV_ERR_CUDA;
  }
  return CBEV_OK;
}

template <typename T>
int dev_alloc(T** p, size_t n) {
  *p = nullptr;
  if (n == 0) n = 1;
  cudaError_t e = cudaMalloc((void**)p, n * sizeof(T));
  if (e != cudaSuccess) {
    cbev_set_error("cudaMalloc(%zu bytes) failed: %s", n * sizeof(T), cudaGetErrorString(e));
    return CBEV_ERR_NOMEM;
  }
  return cudaMemset(*p, 0, n * sizeof(T)) == cudaSuccess ? CBEV_OK : CBEV_ERR_CUDA;
}

template <typename T>
int dev_upload(T** p, const T* host, size_t n) {
  int rc = dev_alloc(p, n);
  if (rc) return rc;
  if (n && host) {
    if (cudaMemcpy(*p, host, n * sizeof(T), cudaMemcpyHostToDevice) != cudaSuccess) {
      cbev_set_error("cudaMemcpy H2D failed");
      return CBEV_ERR_CUDA;
    }
  }
  return CBEV_OK;
}

template <typename T>
void dev_free(T*& p) {
  if (p) cudaFree((void*)p);
  p = nullptr;
}

void free_state(EnvState& s);

void free_pool(PoolDev& p) {
  dev_free(p.ego_state0); dev_free(p.ego_target_speed); dev_free(p.len_ego_route); dev_free(p.ego_tidx0);
  dev_free(p.num_vehicles); dev_free(p.ego_off); dev_free(p.rew_off); dev_free(p.actor_off); dev_free(p.tl_off);
  dev_free(p.ego_cx); dev_free(p.ego_cy); dev_free(p.ego_cyaw); dev_free(p.rew_rx); dev_free(p.rew_ry);
  dev_free(p.rew_cum); dev_free(p.act_kind); dev_free(p.act_beh); dev_free(p.act_state0); dev_free(p.act_cruise_px);
  dev_free(p.act_cruise_mps); dev_free(p.act_beh_p); dev_free(p.act_tidx0); dev_free(p.act_route_off);
  dev_free(p.act_raw_off); dev_free(p.act_retreat_slot); dev_free(p.act_cx); dev_free(p.act_cy); dev_free(p.act_cyaw);
  dev_free(p.act_raw_x); dev_free(p.act_raw_y); dev_free(p.tl_rect); dev_free(p.tl_color); dev_free(p.sg_mat);
  dev_free(p.traj); dev_free(p.traj_off);
  free_state(p.roll);
  p = PoolDev();
}

void free_state(EnvState& s) {
  dev_free(s.scene); dev_free(s.episode); dev_free(s.done); dev_free(s.ego); dev_free(s.egoi);
  dev_free(s.tgt_vis); dev_free(s.stats); dev_free(s.ax); dev_free(s.ay); dev_free(s.ayaw); dev_free(s.av);
  dev_free(s.atarget_mps); dev_free(s.aelapsed); dev_free(s.astate_elapsed); dev_free(s.atidx); dev_free(s.arxlen);
  dev_free(s.aflags); dev_free(s.retreat); dev_free(s.retreat_n);
  s = EnvState();
}

int channels_of(int mask_mode) {
  static const int ch[6] = {1, 2, 4, 5, 6, 7};
  return (mask_mode >= 0 && mask_mode < 6) ? ch[mask_mode] : -1;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int build_tensor_map(cbev_engine* e) {
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || fn == nullptr) {
    cbev_set_error("cuTensorMapEncodeTiled is not available from the driver");
    return CBEV_ERR_CUDA;
  }
  cuuint64_t dims[2] = {(cuuint64_t)e->map_w, (cuuint64_t)e->map_h};
  cuuint64_t strides[1] = {(cuuint64_t)e->map_w};
  cuuint32_t estr[2] = {1, 1};
  // two views of the same map: the one-box fetch window of k_render, and the strip box of k_render_any
  for (int which = 0; which < 2; ++which) {
    cuuint32_t box[2] = {(cuuint32_t)(which ? CBEV_ANY_BOX_W : CBEV_TILE_W),
                         (cuuint32_t)(which ? e->any_box_h : CBEV_TILE_H)};  // sim.cu:compute_view
    CUresult r = ((EncodeTiledFn)fn)(reinterpret_cast<CUtensorMap*>(which ? e->tmap_any : e->tmap),
                                     CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, e->map, dims, strides, box, estr,
                                     CU_TENSOR_MAP_INTERLEAVE_NONE,
                                     which ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                                     CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      cbev_set_error("cuTensorMapEncodeTiled failed with CUresult %d (map %dx%d, box %dx%d)", (int)r, e->map_w, e->map_h,
                     (int)box[0], (int)box[1]);
      return CBEV_ERR_CUDA;
    }
  }
  return CBEV_OK;
}

}  // namespace

// Every entry point runs on the engine's device, whatever the caller's current device is (one engine = one GPU).
static int use_device(cbev_handle e) {
  if (!e) { cbev_set_error("null handle"); return CBEV_ERR_ARG; }
  int cur = -1;
  if (cudaGetDevice(&cur) != cudaSuccess || cur != e->device) CU_TRY(cudaSetDevice(e->device));
  return CBEV_OK;
}

// Second half of a pool change (cbev_upload_scene_pool / cbev_generate_scenes): per-env buffers that depend on the
// pool, the open-loop trajectory tables, and the swap.  `d` is complete on entry and is freed on failure.
static int install_pool(cbev_engine* e, PoolDev& d, const int32_t* actor_off_host, bool live) {
  const int n = d.n_scenes;
  const size_t na = (size_t)d.n_actors_total;
  const int max_retreat = d.max_retreat, max_tl = d.max_tl;
  int rc = 0;
  // ---- per-env buffers that depend on the pool ----
  const size_t Rn = (size_t)(max_retreat ? max_retreat : 1), Ro = (size_t)(e->pool.max_retreat ? e->pool.max_retreat : 1);
  const int32_t new_max_rects = e->cfg.max_actors + CBEV_MAX_TARGETS + max_tl + 1;
  uint32_t* rects = nullptr;
  double* retreat = nullptr;
  int32_t* retreat_n = nullptr;
  const bool grow_rects = !e->rects || new_max_rects > e->max_rects;
  const bool grow_retreat = !e->st.retreat || !live || Rn != Ro;
  if (grow_rects) rc |= dev_alloc(&rects, (size_t)e->N * CBEV_RECT_WORDS * new_max_rects);
  if (grow_retreat) {
    rc |= dev_alloc(&retreat, (size_t)e->N * Rn * 3 * CBEV_SG_MAX);
    rc |= dev_alloc(&retreat_n, (size_t)e->N * Rn);
    if (!rc && live && e->st.retreat) {  // running envs keep the retreat routes they are following (new row stride)
      const size_t row_o = Ro * 3 * CBEV_SG_MAX * sizeof(double), row_n = Rn * 3 * CBEV_SG_MAX * sizeof(double);
      if (cudaMemcpy2D(retreat, row_n, e->st.retreat, row_o, row_o, (size_t)e->N, cudaMemcpyDeviceToDevice) != cudaSuccess ||
          cudaMemcpy2D(retreat_n, Rn * sizeof(int32_t), e->st.retreat_n, Ro * sizeof(int32_t), Ro * sizeof(int32_t),
                       (size_t)e->N, cudaMemcpyDeviceToDevice) != cudaSuccess) {
        cbev_set_error("copying the retreat routes failed");
        rc = CBEV_ERR_CUDA;
      }
    }
  }
  // ---- open-loop actor trajectories: roll every scene out once on the device (k_rollout) ----
  int T = live ? e->pool.traj_steps : e->cfg.trajectory_steps;  // the hand-over step never moves under running envs
  if (!rc && T > 0 && na > 0) {
    const size_t budget = (size_t)4 << 30;  // cap the tables at 4 GiB
    if (!live) {
      while (T > 16 && (size_t)T * na * sizeof(double4) > budget) T /= 2;
    } else if ((size_t)T * na * sizeof(double4) > 2 * budget) {
      cbev_set_error("the extended pool needs %zu bytes of trajectory tables at the %d steps fixed by the first upload",
                     (size_t)T * na * sizeof(double4), T);
      rc = CBEV_ERR_NOMEM;
    }
    std::vector<long long> off((size_t)n);
    long long acc = 0;
    for (int s2 = 0; s2 < n; ++s2) {
      off[s2] = acc;
      acc += (long long)T * (actor_off_host[s2 + 1] - actor_off_host[s2]);
    }
    const size_t S = (size_t)n, A = (size_t)(e->cfg.max_actors > 0 ? e->cfg.max_actors : 1);
    EnvState& r = d.roll;
    if (!rc) {
      rc |= dev_upload(&d.traj_off, off.data(), S);
      rc |= dev_alloc(&d.traj, (size_t)acc);
      rc |= dev_alloc(&r.ax, S * A); rc |= dev_alloc(&r.ay, S * A); rc |= dev_alloc(&r.ayaw, S * A);
      rc |= dev_alloc(&r.av, S * A); rc |= dev_alloc(&r.atarget_mps, S * A); rc |= dev_alloc(&r.aelapsed, S * A);
      rc |= dev_alloc(&r.astate_elapsed, S * A); rc |= dev_alloc(&r.atidx, S * A); rc |= dev_alloc(&r.arxlen, S * A);
      rc |= dev_alloc(&r.aflags, S * A);
      rc |= dev_alloc(&r.retreat, S * Rn * 3 * CBEV_SG_MAX);
      rc |= dev_alloc(&r.retreat_n, S * Rn);
    }
    if (!rc) d.traj_steps = T;
  }
  if (rc) {
    free_pool(d);
    dev_free(rects); dev_free(retreat); dev_free(retreat_n);
    return rc;
  }
  // ---- swap in ----
  free_pool(e->pool);
  e->pool = d;
  if (grow_rects) { dev_free(e->rects); e->rects = rects; e->max_rects = new_max_rects; }
  if (grow_retreat) { dev_free(e->st.retreat); dev_free(e->st.retreat_n); e->st.retreat = retreat; e->st.retreat_n = retreat_n; }
  e->has_pool = true;
  if (!live) e->pool_epoch += 1;  // scene indices may mean something else now: snapshot rows of before are void
  if (e->pool.traj_steps > 0) {
    cbev_launch_rollout(e, 0);
    cudaError_t ce = cudaDeviceSynchronize();
    if (ce != cudaSuccess) {
      cbev_set_error("trajectory roll-out failed: %s", cudaGetErrorString(ce));
      e->has_pool = false;
      return CBEV_ERR_CUDA;
    }
  }
  return CBEV_OK;
}

extern "C" {

int cbev_version(void) { return CBEV_VERSION; }
const char* cbev_last_error(void) { return g_err; }

// OpenCV computeResizeAreaTab for one axis (modules/imgproc/src/resize.cpp, 4.x): for every destination index the
// source taps it covers and their float32 weights, in OpenCV's order.  Checked against cv2 itself in
// tests/test_oracle_contracts.py through the oracle's identical table (oracle/raster.py:_area_table).
static void area_table(int ssize, int dsize, std::vector<int32_t>& off, std::vector<int32_t>& si,
                       std::vector<float>& alpha) {
  const double scale = (double)ssize / dsize;
  off.assign(1, 0);
  for (int dx = 0; dx < dsize; ++dx) {
    const double fsx1 = dx * scale, fsx2 = fsx1 + scale;
    const double cell = std::min(scale, ssize - fsx1);
    int sx1 = (int)std::ceil(fsx1), sx2 = (int)std::floor(fsx2);
    sx2 = std::min(sx2, ssize - 1);
    sx1 = std::min(sx1, sx2);
    if (sx1 - fsx1 > 1e-3) { si.push_back(sx1 - 1); alpha.push_back((float)((sx1 - fsx1) / cell)); }
    for (int sx = sx1; sx < sx2; ++sx) { si.push_back(sx); alpha.push_back((float)(1.0 / cell)); }
    if (fsx2 - sx2 > 1e-3) {
      si.push_back(sx2);
      alpha.push_back((float)(std::min(std::min(fsx2 - sx2, 1.0), cell) / cell));
    }
    off.push_back((int32_t)si.size());
  }
}

// One axis of cv::resize's bilinear set-up in area mode (the dx loop of cv::resize, imgproc/src/resize.cpp): source
// index and the two 11-bit fixed-point taps.  INTER_AREA takes this branch when an axis enlarges (size 64 -> 96).
// Checked against cv2 itself through the oracle's identical table (oracle/raster.py:_linear_area_tab).
static void linear_area_table(int ssize, int dsize, std::vector<int32_t>& ofs, std::vector<int32_t>& a0,
                              std::vector<int32_t>& a1) {
  const double scale = (double)ssize / dsize, inv = 1.0 / scale;
  for (int dx = 0; dx < dsize; ++dx) {
    int sx = (int)std::floor(dx * scale);
    float fx = (float)((dx + 1) - (sx + 1) * inv);
    fx = fx <= 0 ? 0.f : fx - std::floor(fx);
    if (sx >= ssize - 1) { fx = 0.f; sx = ssize - 1; }
    ofs.push_back(sx);
    a0.push_back((int32_t)std::lrintf((1.f - fx) * 2048.f));
    a1.push_back((int32_t)std::lrintf(fx * 2048.f));
  }
}

// area:     rs_tab = [nx, ny, xoff[ow+1], yoff[oh+1], xsi[nx], ysi[ny], xalpha[nx], yalpha[ny],
//                     fxlo[ow], fxhi[ow], fylo[oh], fyhi[oh]]  (first / last source column and row of every output)
// bilinear: rs_tab = [0, 0, xofs[ow], yofs[oh], xa0[ow], xa1[ow], yb0[oh], yb1[oh]]
static int build_resize_tables(cbev_engine* e) {
  const int S = e->cfg.fov_size, oh = e->cfg.obs_h, ow = e->cfg.obs_w;
  e->rs_words = 0;
  if (e->cfg.obs_mode == CBEV_OBS_RGB) { e->rs_mode = CBEV_RS_FAST96; return CBEV_OK; }
  if (oh > S || ow > S) {
    e->rs_mode = CBEV_RS_LINEAR;
    std::vector<int32_t> xo, xa0, xa1, yo, yb0, yb1, tab(2, 0);
    linear_area_table(S, ow, xo, xa0, xa1);
    linear_area_table(S, oh, yo, yb0, yb1);
    // tab[0] = 1: every pair of taps sums to 2048, so four equal texels give their own colour (k_render_any's shortcut)
    bool unit = true;
    for (size_t i = 0; i < xa0.size(); ++i) unit = unit && xa0[i] + xa1[i] == 2048;
    for (size_t i = 0; i < yb0.size(); ++i) unit = unit && yb0[i] + yb1[i] == 2048;
    tab[0] = unit ? 1 : 0;
    for (auto* v : {&xo, &yo, &xa0, &xa1, &yb0, &yb1}) tab.insert(tab.end(), v->begin(), v->end());
    e->rs_words = (int32_t)tab.size();
    return dev_upload(&e->rs_tab, tab.data(), tab.size());
  }
  if (S == 128 && oh == 96 && ow == 96) e->rs_mode = CBEV_RS_FAST96;  // k_render; the tables serve debug flag 256
  else if (oh == S && ow == S) e->rs_mode = CBEV_RS_COPY;
  else if (2 * oh == S && 2 * ow == S) e->rs_mode = CBEV_RS_HALF;
  else e->rs_mode = CBEV_RS_TABLE;
  std::vector<int32_t> xo, yo, xs, ys;
  std::vector<float> xa, ya;
  area_table(S, ow, xo, xs, xa);
  area_table(S, oh, yo, ys, ya);
  std::vector<int32_t> tab;
  tab.push_back((int32_t)xs.size());
  tab.push_back((int32_t)ys.size());
  tab.insert(tab.end(), xo.begin(), xo.end());
  tab.insert(tab.end(), yo.begin(), yo.end());
  tab.insert(tab.end(), xs.begin(), xs.end());
  tab.insert(tab.end(), ys.begin(), ys.end());
  for (float a : xa) { int32_t b; memcpy(&b, &a, 4); tab.push_back(b); }
  for (float a : ya) { int32_t b; memcpy(&b, &a, 4); tab.push_back(b); }
  for (int d = 0; d < ow; ++d) tab.push_back(xs[xo[d]]);
  for (int d = 0; d < ow; ++d) tab.push_back(xs[xo[d + 1] - 1]);
  for (int d = 0; d < oh; ++d) tab.push_back(ys[yo[d]]);
  for (int d = 0; d < oh; ++d) tab.push_back(ys[yo[d + 1] - 1]);
  e->rs_words = (int32_t)tab.size();
  return dev_upload(&e->rs_tab, tab.data(), tab.size());
}

int cbev_create(const cbev_config* cfg, cbev_handle* out) {
  if (!cfg || !out) { cbev_set_error("null argument"); return CBEV_ERR_ARG; }
  *out = nullptr;
  if (cfg->num_envs < 1) { cbev_set_error("num_envs must be >= 1"); return CBEV_ERR_ARG; }
  if (cfg->fov_size != 64 && cfg->fov_size != 128 && cfg->fov_size != 256) {
    // the unmodified reference cannot reset at 512 / 1024 either ("hero_on_obstacle": its scene generators keep the
    // 128-scale coordinates, quirk C-11); a 512-px view would also need a banded raster kernel
    cbev_set_error("size must be 64, 128 or 256 (Town01 map scales the reference can reset on), got %d", cfg->fov_size);
    return CBEV_ERR_ARG;
  }
  if (cfg->obs_mode < 0 || cfg->obs_mode > 3) { cbev_set_error("bad obs_mode %d", cfg->obs_mode); return CBEV_ERR_ARG; }
  const bool masks = cfg->obs_mode == CBEV_OBS_SEMANTIC || cfg->obs_mode == CBEV_OBS_SEMANTIC_U8;
  if (cfg->obs_mode != CBEV_OBS_RGB) {
    // ResizeObservation = cv2.resize(INTER_AREA) of the size x size frame (enlarging takes OpenCV's bilinear branch);
    // every channel plane is streamed with 16-byte stores: 4 float32 masks, or 16 bytes (gray levels, uint8 masks)
    const int px = cfg->obs_h * cfg->obs_w;
    const int mult = cfg->obs_mode == CBEV_OBS_SEMANTIC ? 4 : 16;
    if (cfg->obs_h < 8 || cfg->obs_w < 8 || cfg->obs_h > 256 || cfg->obs_w > 256 || px % mult != 0) {
      cbev_set_error("obs_size must be within 8..256 per side with height*width a multiple of %d (%s), got (%d, %d)",
                     mult, mult == 4 ? "float32 masks" : "16-byte stores of uint8 planes", cfg->obs_h, cfg->obs_w);
      return CBEV_ERR_ARG;
    }
  }
  if (masks && channels_of(cfg->mask_mode) < 0) { cbev_set_error("bad mask_mode %d", cfg->mask_mode); return CBEV_ERR_ARG; }
  if (cfg->frame_stack < 1) { cbev_set_error("frame_stack must be >= 1"); return CBEV_ERR_ARG; }
  if (!(cfg->anchor_x_frac >= 0.0 && cfg->anchor_x_frac <= 1.0 && cfg->anchor_y_frac >= 0.0 && cfg->anchor_y_frac <= 1.0)) {
    cbev_set_error("ego anchor fractions must be within [0, 1]");
    return CBEV_ERR_ARG;
  }
  const int F = cfg->obs_mode == CBEV_OBS_RGB ? 1 : cfg->frame_stack;
  if (F > 1 && cfg->ring_slots < 2 * F - 1) { cbev_set_error("ring_slots must be >= 2*frame_stack-1 (%d), got %d", 2 * F - 1, cfg->ring_slots); return CBEV_ERR_ARG; }
  if (F == 1 && cfg->ring_slots < 1) { cbev_set_error("ring_slots must be >= 1"); return CBEV_ERR_ARG; }
  if (cfg->action_mode == CBEV_ACTION_DISCRETE && (cfg->n_discrete < 1 || cfg->n_discrete > 16)) { cbev_set_error("n_discrete must be in [1, 16]"); return CBEV_ERR_ARG; }
  if (cfg->max_actors < 0) { cbev_set_error("max_actors must be >= 0"); return CBEV_ERR_ARG; }

  cbev_engine* e = new (std::nothrow) cbev_engine();
  if (!e) return CBEV_ERR_NOMEM;
  e->cfg = *cfg;
  e->cfg.frame_stack = F;
  if (F == 1) e->cfg.ring_slots = 1;
  e->N = cfg->num_envs;
  cudaGetDevice(&e->device);
  // FovRenderer constants (envs/fov.py:30-44); padding = crop_size (envs/world.py:69-78)
  const int m = cfg->fov_size - 1;
  int ax = (int)nearbyint((double)m * cfg->anchor_x_frac), ay = (int)nearbyint((double)m * cfg->anchor_y_frac);
  ax = ax < 0 ? 0 : (ax > m ? m : ax);
  ay = ay < 0 ? 0 : (ay > m ? m : ay);
  e->anchor_x = ax;
  e->anchor_y = ay;
  int mx = ax > m - ax ? ax : m - ax, my = ay > m - ay ? ay : m - ay;
  int crop = (int)ceil(2.0 * hypot((double)mx, (double)my));
  if (crop < cfg->fov_size) crop = cfg->fov_size;
  e->crop = crop;  // any size: the raster kernel only ever fetches the window a frame can sample
  e->pad = crop;
  {
    // fetch window of one frame: <= ceil(S * sqrt(2)) + 2 px on a side (sim.cu:compute_view).  k_render_any lands it as
    // column strips of CBEV_ANY_BOX_W bytes (15 bytes of TMA alignment slack) x row boxes of <= 256 rows.
    const int S = cfg->fov_size;
    const int win = (int)ceil(S * sqrt(2.0)) + 2;
    const int tile_h = (win + 7) & ~7;
    e->any_nby = (tile_h + 255) / 256;
    e->any_box_h = ((tile_h + e->any_nby - 1) / e->any_nby + 7) & ~7;
    e->any_nbx = (win + 15 + CBEV_ANY_BOX_W - 1) / CBEV_ANY_BOX_W;
    e->win_max = S == 128 ? CBEV_TILE_H : e->any_box_h * e->any_nby;
  }
  e->channels = masks ? channels_of(cfg->mask_mode) : 1;
  if (cfg->obs_mode == CBEV_OBS_SEMANTIC) e->frame_bytes = (int64_t)e->channels * cfg->obs_h * cfg->obs_w * 4;
  else if (cfg->obs_mode == CBEV_OBS_SEMANTIC_U8) e->frame_bytes = (int64_t)e->channels * cfg->obs_h * cfg->obs_w;
  else if (cfg->obs_mode == CBEV_OBS_GRAY) e->frame_bytes = (int64_t)cfg->obs_h * cfg->obs_w;
  else e->frame_bytes = (int64_t)cfg->fov_size * cfg->fov_size * 3;

  const size_t N = (size_t)e->N, A = (size_t)(cfg->max_actors > 0 ? cfg->max_actors : 1);
  int rc = 0;
  rc |= dev_alloc(&e->st.scene, N);
  rc |= dev_alloc(&e->st.episode, N);
  rc |= dev_alloc(&e->st.done, N);
  rc |= dev_alloc(&e->st.ego, N * 24);
  rc |= dev_alloc(&e->st.egoi, N * 8);
  rc |= dev_alloc(&e->st.tgt_vis, N * CBEV_TGT_WORDS);
  rc |= dev_alloc(&e->st.stats, N * 12);
  rc |= dev_alloc(&e->st.ax, N * A);
  rc |= dev_alloc(&e->st.ay, N * A);
  rc |= dev_alloc(&e->st.ayaw, N * A);
  rc |= dev_alloc(&e->st.av, N * A);
  rc |= dev_alloc(&e->st.atarget_mps, N * A);
  rc |= dev_alloc(&e->st.aelapsed, N * A);
  rc |= dev_alloc(&e->st.astate_elapsed, N * A);
  rc |= dev_alloc(&e->st.atidx, N * A);
  rc |= dev_alloc(&e->st.arxlen, N * A);
  rc |= dev_alloc(&e->st.aflags, N * A);
  rc |= dev_alloc(&e->desc, N * CBEV_DESC_WORDS);
  rc |= dev_alloc(&e->order, N);
  rc |= dev_alloc(&e->order_cnt, (size_t)2);
  rc |= dev_alloc(&e->move_order, N);
  rc |= dev_alloc(&e->move_cnt, (size_t)2);
  rc |= dev_alloc(&e->fov, N * (size_t)cfg->fov_size * cfg->fov_size);
  rc |= dev_alloc(&e->gstats, (size_t)CBEV_STATS_FIELDS);
  rc |= build_resize_tables(e);
  rc |= dev_alloc((uint8_t**)&e->h_reward_dev, N * 10);  // one block: reward f64[N] | terminated u8[N] | truncated u8[N]
  e->h_term_dev = (uint8_t*)e->h_reward_dev + N * 8;
  e->h_trunc_dev = e->h_term_dev + N;
  rc |= dev_alloc((uint8_t**)&e->h_actions_dev, N * 16);
  if (rc) { cbev_destroy(e); return rc; }
  cudaMemset(e->st.scene, 0xff, N * sizeof(int32_t));
  {  // identifies the engine in its snapshot rows
    uint64_t z = (uint64_t)std::chrono::steady_clock::now().time_since_epoch().count() ^ (uint64_t)(uintptr_t)e;
    try {
      std::random_device rd;
      z ^= ((uint64_t)rd() << 32) | (uint64_t)rd();
    } catch (...) {
    }
    z += 0x9E3779B97F4A7C15ull;  // splitmix64 finaliser
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    e->token = z ^ (z >> 31);
  }
  *out = e;
  return CBEV_OK;
}

int cbev_destroy(cbev_handle e) {
  if (!e) return CBEV_OK;
  use_device(e);
  free_pool(e->pool);
  free_state(e->st);
  free_state(e->branch);
  dev_free(e->br_stage_desc); dev_free(e->br_stage_rects); dev_free(e->br_desc); dev_free(e->br_rects);
  dev_free(e->br_window);
  dev_free(e->fov_mask); dev_free(e->rs_tab); dev_free(e->trace);
  dev_free(e->order); dev_free(e->order_cnt); dev_free(e->move_order); dev_free(e->move_cnt);
  dev_free(e->map); dev_free(e->desc); dev_free(e->rects); dev_free(e->fov); dev_free(e->gstats);
  dev_free(e->h_reward_dev);
  { uint8_t* p = (uint8_t*)e->h_actions_dev; dev_free(p); }
  if (e->side_stream) cudaStreamDestroy(e->side_stream);
  if (e->ev_sim) cudaEventDestroy(e->ev_sim);
  if (e->ev_copy) cudaEventDestroy(e->ev_copy);
  if (e->ev_judge) cudaEventDestroy(e->ev_judge);
  if (e->prof_ev) {
    for (int i = 0; i < CBEV_PROF_EVENTS * CBEV_PROF_MAX; ++i) cudaEventDestroy(e->prof_ev[i]);
    delete[] e->prof_ev;
  }
  delete e;
  return CBEV_OK;
}

int cbev_upload_map(cbev_handle e, const uint8_t* cls_host, int32_t w, int32_t h_px) {
  if (!e || !cls_host) { cbev_set_error("null argument"); return CBEV_ERR_ARG; }
  { int rc0 = use_device(e); if (rc0) return rc0; }
  if (w < 16 || h_px < 16 || (w % 16) != 0) { cbev_set_error("map width must be a multiple of 16 (TMA row pitch), got %dx%d", w, h_px); return CBEV_ERR_ARG; }
  for (size_t i = 0; i < (size_t)w * h_px; ++i)
    if (cls_host[i] > 2) { cbev_set_error("map classes must be 0 (non-drivable), 1 (drivable) or 2 (sidewalk)"); return CBEV_ERR_ARG; }
  dev_free(e->map);
  int rc = dev_upload(&e->map, cls_host, (size_t)w * h_px);
  if (rc) return rc;
  e->map_w = w;
  e->map_h = h_px;
  rc = build_tensor_map(e);
  if (rc) return rc;
  e->has_map = true;
  return CBEV_OK;
}

int cbev_upload_scene_pool(cbev_handle e, const cbev_pool_desc* p) {
  if (!e || !p) { cbev_set_error("null argument"); return CBEV_ERR_ARG; }
  { int rc0 = use_device(e); if (rc0) return rc0; }
  if (p->n_scenes < 1) { cbev_set_error("scene pool is empty"); return CBEV_ERR_ARG; }
  const int n = p->n_scenes;
  // ---- validate (the reference raises on malformed scenes at reset; here at upload) ----
  int max_actors = 0, max_targets = 0, max_tl = 0, max_retreat = 0;
  std::vector<int32_t> slots((size_t)(p->n_actors_total > 0 ? p->n_actors_total : 1), -1);
  for (int s = 0; s < n; ++s) {
    int nt = p->ego_off[s + 1] - p->ego_off[s];
    if (nt < 2 || nt > CBEV_MAX_TARGETS) { cbev_set_error("scene %d: ego route has %d points, supported range is [2, %d]", s, nt, CBEV_MAX_TARGETS); return CBEV_ERR_ARG; }
    if (p->ego_tidx0[s] < 0 || p->ego_tidx0[s] >= nt) { cbev_set_error("scene %d: ego target index out of range", s); return CBEV_ERR_ARG; }
    int a0 = p->actor_off[s], a1 = p->actor_off[s + 1];
    if (a1 < a0 || a1 > p->n_actors_total) { cbev_set_error("scene %d: bad actor offsets", s); return CBEV_ERR_ARG; }
    int nret = 0;
    bool seen_ped = false;
    for (int a = a0; a < a1; ++a) {
      if (p->act_kind[a] > 1) { cbev_set_error("scene %d: bad actor kind", s); return CBEV_ERR_ARG; }
      if (p->act_kind[a] == 1) seen_ped = true;
      else if (seen_ped) { cbev_set_error("scene %d: vehicles must precede pedestrians (draw / collision order)", s); return CBEV_ERR_ARG; }
      int np = p->act_route_off[a + 1] - p->act_route_off[a];
      if (np < 2) { cbev_set_error("scene %d: actor route needs >= 2 points", s); return CBEV_ERR_ARG; }
      if (p->act_beh[a] > CBEV_BEH_STOP_RETURN) { cbev_set_error("scene %d: unknown behaviour id %d", s, p->act_beh[a]); return CBEV_ERR_ARG; }
      if (p->act_beh[a] == CBEV_BEH_STOP_RETURN) {
        if (!p->sg_mat) { cbev_set_error("scene %d: StopReturn behaviour needs sg_mat (retreat smoothing operators)", s); return CBEV_ERR_ARG; }
        int nr = p->act_raw_off[a + 1] - p->act_raw_off[a];
        if (nr + 1 > CBEV_SG_MAX) { cbev_set_error("scene %d: retreat route of %d points exceeds CBEV_SG_MAX", s, nr + 1); return CBEV_ERR_ARG; }
        slots[a] = nret++;
      }
    }
    if (a1 - a0 > max_actors) max_actors = a1 - a0;
    if (nt > max_targets) max_targets = nt;
    int ntl = p->tl_off[s + 1] - p->tl_off[s];
    if (ntl > max_tl) max_tl = ntl;
    if (nret > max_retreat) max_retreat = nret;
  }
  if (max_actors > e->cfg.max_actors) { cbev_set_error("pool has scenes with %d actors but the engine was created with max_actors=%d", max_actors, e->cfg.max_actors); return CBEV_ERR_ARG; }

  // Environments may be mid-episode (SyncVectorEnv resets a subset with a new scene while the others keep running):
  // a pool uploaded then must EXTEND the previous one (scene i keeps its index), and everything a running env
  // depends on stays as it is -- the length of the trajectory tables (the hand-over step), the per-env retreat
  // routes and their row stride.  The new pool is built on the side and swapped in only when complete, so a failed
  // upload leaves the previous pool in place.
  const bool live = e->was_reset && e->has_pool;
  if (live) {
    if (n < e->pool.n_scenes) { cbev_set_error("a pool uploaded while environments are running must extend the previous one (%d scenes < %d)", n, e->pool.n_scenes); return CBEV_ERR_ARG; }
    CU_TRY(cudaDeviceSynchronize());
    if (max_retreat < e->pool.max_retreat) max_retreat = e->pool.max_retreat;
  }
  PoolDev d;
  d.n_scenes = n;
  d.n_actors_total = p->n_actors_total;
  d.max_actors = max_actors;
  d.max_targets = max_targets;
  d.max_tl = max_tl;
  d.max_retreat = max_retreat;
  const size_t na = (size_t)p->n_actors_total, nr = (size_t)p->ego_off[n], nq = (size_t)p->rew_off[n];
  const size_t npts = na ? (size_t)p->act_route_off[na] : 0, nraw = na ? (size_t)p->act_raw_off[na] : 0;
  const size_t ntl = (size_t)p->tl_off[n];
  int rc = 0;
  rc |= dev_upload(&d.ego_state0, p->ego_state0, (size_t)n * 4);
  rc |= dev_upload(&d.ego_target_speed, p->ego_target_speed, (size_t)n);
  rc |= dev_upload(&d.len_ego_route, p->len_ego_route, (size_t)n);
  rc |= dev_upload(&d.ego_tidx0, p->ego_tidx0, (size_t)n);
  rc |= dev_upload(&d.num_vehicles, p->num_vehicles, (size_t)n);
  rc |= dev_upload(&d.ego_off, p->ego_off, (size_t)n + 1);
  rc |= dev_upload(&d.rew_off, p->rew_off, (size_t)n + 1);
  rc |= dev_upload(&d.actor_off, p->actor_off, (size_t)n + 1);
  rc |= dev_upload(&d.tl_off, p->tl_off, (size_t)n + 1);
  rc |= dev_upload(&d.ego_cx, p->ego_cx, nr);
  rc |= dev_upload(&d.ego_cy, p->ego_cy, nr);
  rc |= dev_upload(&d.ego_cyaw, p->ego_cyaw, nr);
  rc |= dev_upload(&d.rew_rx, p->rew_rx, nq);
  rc |= dev_upload(&d.rew_ry, p->rew_ry, nq);
  rc |= dev_upload(&d.rew_cum, p->rew_cum, nq);
  rc |= dev_upload(&d.act_kind, p->act_kind, na);
  rc |= dev_upload(&d.act_beh, p->act_beh, na);
  rc |= dev_upload(&d.act_state0, p->act_state0, na * 4);
  rc |= dev_upload(&d.act_cruise_px, p->act_cruise_px, na);
  rc |= dev_upload(&d.act_cruise_mps, p->act_cruise_mps, na);
  rc |= dev_upload(&d.act_beh_p, p->act_beh_p, na * 4);
  rc |= dev_upload(&d.act_tidx0, p->act_tidx0, na);
  rc |= dev_upload(&d.act_route_off, p->act_route_off, na + 1);
  rc |= dev_upload(&d.act_raw_off, p->act_raw_off, na + 1);
  rc |= dev_upload(&d.act_retreat_slot, slots.data(), na ? na : 1);
  rc |= dev_upload(&d.act_cx, p->act_cx, npts);
  rc |= dev_upload(&d.act_cy, p->act_cy, npts);
  rc |= dev_upload(&d.act_cyaw, p->act_cyaw, npts);
  rc |= dev_upload(&d.act_raw_x, p->act_raw_x, nraw);
  rc |= dev_upload(&d.act_raw_y, p->act_raw_y, nraw);
  rc |= dev_upload(&d.tl_rect, p->tl_rect, ntl * 4);
  rc |= dev_upload(&d.tl_color, p->tl_color, ntl);
  if (p->sg_mat) rc |= dev_upload(&d.sg_mat, p->sg_mat, (size_t)(CBEV_SG_MAX + 1) * CBEV_SG_MAX * CBEV_SG_MAX);
  if (rc) { free_pool(d); return rc; }
  return install_pool(e, d, p->actor_off, live);
}

// Device-side generation of scripted scenes: see include/cbev.h.
int cbev_generate_scenes(cbev_handle e, int32_t n, const uint8_t* kinds, const int32_t* levels, const int64_t* seeds,
                         const double* sg_mat, int32_t* attempts_host) {
  if (!e || !kinds || !levels || !seeds || !sg_mat) { cbev_set_error("null argument"); return CBEV_ERR_ARG; }
  { int rc0 = use_device(e); if (rc0) return rc0; }
  if (!e->has_map) { cbev_set_error("no map uploaded (cbev_upload_map): spawn validation needs it"); return CBEV_ERR_STATE; }
  if (n < 1) { cbev_set_error("scene pool is empty"); return CBEV_ERR_ARG; }
  // the layout of a scripted scene is a function of (kind, level): actors and route lengths are known up front
  std::vector<int32_t> ego_off(n + 1), rew_off(n + 1), actor_off(n + 1), tl_off(n + 1, 0), route_off(1, 0), raw_off(1, 0), slots;
  int max_actors = 0, max_retreat = 0;
  for (int s = 0; s < n; ++s) {
    const int lv = levels[s];
    if ((kinds[s] != 1 && kinds[s] != 2) || lv < 1 || lv > 4 || (kinds[s] == 1 && lv > 3) || seeds[s] < 0) {
      cbev_set_error("scene %d: kind must be 1 (lead_brake, levels 1-3) or 2 (jaywalk, levels 1-4) and the seed >= 0", s);
      return CBEV_ERR_ARG;
    }
    ego_off[s] = 6 * s; rew_off[s] = 6 * s; actor_off[s] = (int32_t)slots.size();
    int nret = 0;
    auto add = [&](int pts, bool retreat) {
      route_off.push_back(route_off.back() + pts);
      raw_off.push_back(raw_off.back() + pts);
      slots.push_back(retreat ? nret++ : -1);
    };
    if (kinds[s] == 1) {            // lead_brake.py: lead (6) [+ left lane (7)] [+ rear (6)]
      add(6, false);
      if (lv >= 2) add(7, false);
      if (lv >= 3) add(6, false);
    } else {                        // jaywalk.py: [rear vehicle (6) at level 4] + pedestrian (8); StopReturn from level 3
      if (lv >= 4) add(6, false);
      add(8, lv >= 3);
    }
    max_actors = std::max(max_actors, (int)slots.size() - actor_off[s]);
    max_retreat = std::max(max_retreat, nret);
  }
  ego_off[n] = rew_off[n] = 6 * n;
  actor_off[n] = (int32_t)slots.size();
  if (max_actors > e->cfg.max_actors) { cbev_set_error("generated scenes have up to %d actors but the engine was created with max_actors=%d", max_actors, e->cfg.max_actors); return CBEV_ERR_ARG; }
  const bool live = e->was_reset && e->has_pool;
  if (live) {
    if (n < e->pool.n_scenes) { cbev_set_error("a pool generated while environments are running must extend the previous one"); return CBEV_ERR_ARG; }
    CU_TRY(cudaDeviceSynchronize());
    if (max_retreat < e->pool.max_retreat) max_retreat = e->pool.max_retreat;
  }
  const size_t na = slots.size(), npts = (size_t)route_off.back();
  PoolDev d;
  d.n_scenes = n; d.n_actors_total = (int32_t)na; d.max_actors = max_actors; d.max_targets = 6; d.max_tl = 0;
  d.max_retreat = max_retreat;
  int rc = 0;
  rc |= dev_alloc(&d.ego_state0, (size_t)n * 4); rc |= dev_alloc(&d.ego_target_speed, (size_t)n);
  rc |= dev_alloc(&d.len_ego_route, (size_t)n); rc |= dev_alloc(&d.ego_tidx0, (size_t)n);
  rc |= dev_alloc(&d.num_vehicles, (size_t)n);
  rc |= dev_upload(&d.ego_off, ego_off.data(), (size_t)n + 1); rc |= dev_upload(&d.rew_off, rew_off.data(), (size_t)n + 1);
  rc |= dev_upload(&d.actor_off, actor_off.data(), (size_t)n + 1); rc |= dev_upload(&d.tl_off, tl_off.data(), (size_t)n + 1);
  rc |= dev_alloc(&d.ego_cx, (size_t)6 * n); rc |= dev_alloc(&d.ego_cy, (size_t)6 * n); rc |= dev_alloc(&d.ego_cyaw, (size_t)6 * n);
  rc |= dev_alloc(&d.rew_rx, (size_t)6 * n); rc |= dev_alloc(&d.rew_ry, (size_t)6 * n); rc |= dev_alloc(&d.rew_cum, (size_t)6 * n);
  rc |= dev_alloc(&d.act_kind, na); rc |= dev_alloc(&d.act_beh, na); rc |= dev_alloc(&d.act_state0, na * 4);
  rc |= dev_alloc(&d.act_cruise_px, na); rc |= dev_alloc(&d.act_cruise_mps, na); rc |= dev_alloc(&d.act_beh_p, na * 4);
  rc |= dev_alloc(&d.act_tidx0, na);
  rc |= dev_upload(&d.act_route_off, route_off.data(), na + 1); rc |= dev_upload(&d.act_raw_off, raw_off.data(), na + 1);
  rc |= dev_upload(&d.act_retreat_slot, slots.data(), na);
  rc |= dev_alloc(&d.act_cx, npts); rc |= dev_alloc(&d.act_cy, npts); rc |= dev_alloc(&d.act_cyaw, npts);
  rc |= dev_alloc(&d.act_raw_x, npts); rc |= dev_alloc(&d.act_raw_y, npts);
  rc |= dev_alloc(&d.tl_rect, (size_t)4); rc |= dev_alloc(&d.tl_color, (size_t)1);
  rc |= dev_upload(&d.sg_mat, sg_mat, (size_t)(CBEV_SG_MAX + 1) * CBEV_SG_MAX * CBEV_SG_MAX);
  uint8_t* kinds_d = nullptr;
  int32_t *levels_d = nullptr, *att_d = nullptr;
  long long* seeds_d = nullptr;
  rc |= dev_upload(&kinds_d, kinds, (size_t)n); rc |= dev_upload(&levels_d, levels, (size_t)n);
  rc |= dev_upload(&seeds_d, (const long long*)seeds, (size_t)n); rc |= dev_alloc(&att_d, (size_t)n);
  std::vector<int32_t> att((size_t)n, 0);
  if (!rc) {
    cbev_launch_generate(e, d, kinds_d, levels_d, seeds_d, att_d, 0);
    cudaError_t ce = cudaDeviceSynchronize();
    if (ce == cudaSuccess) ce = cudaMemcpy(att.data(), att_d, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost);
    if (ce != cudaSuccess) { cbev_set_error("scene generation failed: %s", cudaGetErrorString(ce)); rc = CBEV_ERR_CUDA; }
  }
  dev_free(kinds_d); dev_free(levels_d); dev_free(seeds_d); dev_free(att_d);
  if (!rc)
    for (int s = 0; s < n; ++s)
      if (att[s] < 0) {  // the reference raises here (carlabev.py:129-131)
        cbev_set_error("Failed to reset into a valid initial state after 10 attempts (scene %d, seed %lld)", s, (long long)seeds[s]);
        rc = CBEV_ERR_ARG;
        break;
      }
  if (attempts_host) memcpy(attempts_host, att.data(), (size_t)n * sizeof(int32_t));
  if (rc) { free_pool(d); return rc; }
  return install_pool(e, d, actor_off.data(), live);
}

int cbev_pool_counts(cbev_handle e, int32_t counts[8]) {
  if (!e || !counts) { cbev_set_error("null argument"); return CBEV_ERR_ARG; }
  { int rc0 = use_device(e); if (rc0) return rc0; }
  if (!e->has_pool) { cbev_set_error("no scene pool"); return CBEV_ERR_STATE; }
  const PoolDev& d = e->pool;
  int32_t last[5] = {0, 0, 0, 0, 0};
  const int n = d.n_scenes, na = d.n_actors_total;
  CU_TRY(cudaMemcpy(&last[0], d.ego_off + n, 4, cudaMemcpyDeviceToHost));
  CU_TRY(cudaMemcpy(&last[1], d.rew_off + n, 4, cudaMemcpyDeviceToHost));
  CU_TRY(cudaMemcpy(&last[2], d.tl_off + n, 4, cudaMemcpyDeviceToHost));
  if (na) {
    CU_TRY(cudaMemcpy(&last[3], d.act_route_off + na, 4, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(&last[4], d.act_raw_off + na, 4, cudaMemcpyDeviceToHost));
  }
  counts[0] = n; counts[1] = na; counts[2] = last[0]; counts[3] = last[1]; counts[4] = last[3]; counts[5] = last[4];
  counts[6] = last[2]; counts[7] = d.traj_steps;
  return CBEV_OK;
}

int cbev_read_scene_pool(cbev_handle e, const cbev_pool_desc* dst) {
  if (!e || !dst) { cbev_set_error("null argument"); return CBEV_ERR_ARG; }
  { int rc0 = use_device(e); if (rc0) return rc0; }
  if (!e->has_pool) { cbev_set_error("no scene pool"); return CBEV_ERR_STATE; }
  int32_t c[8];
  int rc = cbev_pool_counts(e, c);
  if (rc) return rc;
  const PoolDev& d = e->pool;
  const size_t n = (size_t)c[0], na = (size_t)c[1], nr = (size_t)c[2], nq = (size_t)c[3], np = (size_t)c[4], nw = (size_t)c[5],
               ntl = (size_t)c[6];
#define RD(field, count)                                                                                          \
  if (dst->field && (count))                                                                                      \
    CU_TRY(cudaMemcpy((void*)dst->field, d.field, (count) * sizeof(*d.field), cudaMemcpyDeviceToHost));
  RD(ego_state0, n * 4) RD(ego_target_speed, n) RD(ego_tidx0, n) RD(len_ego_route, n) RD(num_vehicles, n)
  RD(ego_off, n + 1) RD(rew_off, n + 1) RD(actor_off, n + 1) RD(tl_off, n + 1)
  RD(ego_cx, nr) RD(ego_cy, nr) RD(ego_cyaw, nr) RD(rew_rx, nq) RD(rew_ry, nq) RD(rew_cum, nq)
  RD(act_kind, na) RD(act_state0, na * 4) RD(act_tidx0, na) RD(act_cruise_px, na) RD(act_cruise_mps, na)
  RD(act_beh, na) RD(act_beh_p, na * 4) RD(act_route_off, na + 1) RD(act_raw_off, na + 1)
  RD(act_cx, np) RD(act_cy, np) RD(act_cyaw, np) RD(act_raw_x, nw) RD(act_raw_y, nw) RD(tl_rect, ntl * 4) RD(tl_color, ntl)
#undef RD
  return CBEV_OK;
}

int64_t cbev_frame_bytes(cbev_handle e) { return e ? e->frame_bytes : -1; }

int cbev_bind_obs_ring(cbev_handle e, void* ring_dev, int64_t bytes) {
  if (!e || !ring_dev) { cbev_set_error("null argument"); return CBEV_ERR_ARG; }
  { int rc0 = use_device(e); if (rc0) return rc0; }
  int64_t need = (int64_t)e->N * e->cfg.ring_slots * e->frame_bytes;
  if (bytes < need) { cbev_set_error("observation ring needs %lld bytes, got %lld", (long long)need, (long long)bytes); return CBEV_ERR_ARG; }
  if (((uintptr_t)ring_dev & 15) != 0) { cbev_set_error("observation ring must be 16-byte aligned"); return CBEV_ERR_ARG; }
  e->ring = ring_dev;
  e->ring_bytes = bytes;
  return CBEV_OK;
}

int cbev_bind_final_obs(cbev_handle e, void* final_dev, int64_t bytes) {
  if (!e) { cbev_set_error("null handle"); return CBEV_ERR_ARG; }
  if (e->cfg.autoreset != CBEV_AUTORESET_SAME_STEP) {
    cbev_set_error("final observations are written only under CBEV_AUTORESET_SAME_STEP (autoreset = %d)", e->cfg.autoreset);
    return CBEV_ERR_ARG;
  }
  if (final_dev) {
    if (((uintptr_t)final_dev & 15) != 0) { cbev_set_error("final observation buffer must be 16-byte aligned"); return CBEV_ERR_ARG; }
    const int64_t need = (int64_t)e->N * e->cfg.frame_stack * e->frame_bytes;
    if (bytes < need) { cbev_set_error("final observation buffer needs %lld bytes (N * F * frame bytes), got %lld", (long long)need, (long long)bytes); return CBEV_ERR_ARG; }
  }
  e->final_obs = final_dev;
  return CBEV_OK;
}

static int check_ready(cbev_handle e, bool need_reset) {
  if (!e) { cbev_set_error("null handle"); return CBEV_ERR_ARG; }
  { int rc0 = use_device(e); if (rc0) return rc0; }
  if (!e->has_map) { cbev_set_error("no map uploaded (cbev_upload_map)"); return CBEV_ERR_STATE; }
  if (!e->has_pool) { cbev_set_error("no scene pool uploaded (cbev_upload_scene_pool)"); return CBEV_ERR_STATE; }
  if (!e->ring) { cbev_set_error("no observation ring bound (cbev_bind_obs_ring)"); return CBEV_ERR_STATE; }
  if (need_reset && !e->was_reset) { cbev_set_error("step() called before reset()"); return CBEV_ERR_STATE; }
  return CBEV_OK;
}

int cbev_reset(cbev_handle e, const uint8_t* mask_dev, const int32_t* scene_ids_dev, void* stream) {
  int rc = check_ready(e, false);
  if (rc) return rc;
  if (!scene_ids_dev) { cbev_set_error("scene_ids is required"); return CBEV_ERR_ARG; }
  if (mask_dev && !e->was_reset) { cbev_set_error("the first reset must cover every env (mask = NULL)"); return CBEV_ERR_STATE; }
  cudaStream_t s = (cudaStream_t)stream;
  const int F = e->cfg.frame_stack, L = e->cfg.ring_slots;
  if (e->head < 0) e->head = F - 1;
  cbev_launch_reset(e, mask_dev, scene_ids_dev, s);
  if ((rc = debug_sync("k_reset", s))) return rc;
  if (cbev_launch_render(e, e->head, F > 1 ? L - F + 1 : 0, s)) return CBEV_ERR_CUDA;  // cbev_launch_render says why
  if ((rc = debug_sync("k_render (reset frame)", s))) return rc;
  CU_TRY(cudaGetLastError());
  e->was_reset = true;
  return CBEV_OK;
}

static int ensure_side_stream(cbev_engine* e) {
  if (e->side_stream) return CBEV_OK;
  int lo = 0, hi = 0;  // numerically lowest = highest priority: k_judge's few CTAs must not queue behind the raster grid
  CU_TRY(cudaDeviceGetStreamPriorityRange(&lo, &hi));
  // (measured with the LEAST priority instead: k_judge's CTAs are then only placed as the raster grid drains, the
  //  raster kernel runs undisturbed at 0.1767 ms but the step ends later, 0.1937 vs 0.1923 ms, and reward / flags
  //  reach the host at the end of the step instead of 90 us into it)
  CU_TRY(cudaStreamCreateWithPriority(&e->side_stream, cudaStreamNonBlocking, hi));
  CU_TRY(cudaEventCreateWithFlags(&e->ev_sim, cudaEventDisableTiming));
  CU_TRY(cudaEventCreateWithFlags(&e->ev_judge, cudaEventDisableTiming));
  CU_TRY(cudaEventCreateWithFlags(&e->ev_copy, cudaEventDisableTiming));
  return CBEV_OK;
}

int cbev_step_ex(cbev_handle e, const void* actions_dev, const cbev_step_out* out, const cbev_host_out* host, void* stream);

int cbev_step(cbev_handle e, const void* actions_dev, const cbev_step_out* out, void* stream) {
  return cbev_step_ex(e, actions_dev, out, nullptr, stream);
}

int cbev_step_ex(cbev_handle e, const void* actions_dev, const cbev_step_out* out, const cbev_host_out* host,
                 void* stream) {
  int rc = check_ready(e, true);
  if (rc) return rc;
  if (!actions_dev || !out || !out->reward || !out->terminated || !out->truncated) { cbev_set_error("actions, reward, terminated and truncated are required"); return CBEV_ERR_ARG; }
  if (host && (!host->reward || !host->terminated || !host->truncated)) { cbev_set_error("null host buffer"); return CBEV_ERR_ARG; }
  if ((rc = ensure_side_stream(e))) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const int F = e->cfg.frame_stack, L = e->cfg.ring_slots;
  int head = e->head + 1;
  if (head >= L) head = F - 1;
  const int mirror = F > 1 ? L - F + 1 : 0;
  // Per step: k_move on `stream`; then k_judge on the (high-priority) side stream CONCURRENTLY with k_render on
  // `stream` -- the raster kernel reads only the descriptor / draw list k_move wrote, the judging chain (reward,
  // termination, statistics) touches neither.  `stream` joins the side stream at the end of the step, so whatever
  // the caller enqueues next (its reads of reward / flags, the next step) is ordered after both.
  // With an action repeat above 1 (or debug flag 1024) k_step_repeat takes the place of k_move and k_judge: it runs
  // every sub-step with its judging, so the side stream carries only the host copies.
  const bool fused = e->action_repeat > 1 || (e->debug_flags & CBEV_DBG_STEP_REPEAT);
  const bool prof = e->profiling && e->prof_n < CBEV_PROF_MAX;
  cudaEvent_t* pe = prof ? e->prof_ev + CBEV_PROF_EVENTS * e->prof_n : nullptr;
  if (prof) cudaEventRecord(pe[0], s);
  if (fused) cbev_launch_step_repeat(e, actions_dev, out, s);
  else cbev_launch_move(e, actions_dev, out, s);
  if (prof) cudaEventRecord(pe[1], s);
  if ((rc = debug_sync(fused ? "k_step_repeat" : "k_move", s))) return rc;
  // debug flag 2 (timing probe): k_judge on the caller's stream, i.e. serial between k_move and k_render
  cudaStream_t js = (e->debug_flags & CBEV_DBG_JUDGE_SERIAL) ? s : e->side_stream;
  if (js != s) {
    CU_TRY(cudaEventRecord(e->ev_sim, s));
    CU_TRY(cudaStreamWaitEvent(js, e->ev_sim, 0));
  }
  if (!fused) {
    if (prof) cudaEventRecord(pe[3], js);
    cbev_launch_judge(e, out, js);
    if (prof) cudaEventRecord(pe[4], js);
    if ((rc = debug_sync("k_judge", js))) return rc;
  }
  if (host) {  // reward / flags are final after k_judge: copy them out while the raster kernel runs
    const size_t N = (size_t)e->N;
    const cbev_host_out* ho = host;
    const bool packed_dev = out->terminated == (uint8_t*)out->reward + N * 8 && out->truncated == out->terminated + N;
    const bool packed_host = ho->terminated == (uint8_t*)ho->reward + N * 8 && ho->truncated == ho->terminated + N;
    if (packed_dev && packed_host) {
      // both sides laid the three outputs out back to back: one D2H copy instead of three
      CU_TRY(cudaMemcpyAsync(ho->reward, out->reward, N * 10, cudaMemcpyDeviceToHost, js));
    } else {
      CU_TRY(cudaMemcpyAsync(ho->reward, out->reward, N * 8, cudaMemcpyDeviceToHost, js));
      CU_TRY(cudaMemcpyAsync(ho->terminated, out->terminated, N, cudaMemcpyDeviceToHost, js));
      CU_TRY(cudaMemcpyAsync(ho->truncated, out->truncated, N, cudaMemcpyDeviceToHost, js));
    }
    if (ho->cause && out->cause) CU_TRY(cudaMemcpyAsync(ho->cause, out->cause, N, cudaMemcpyDeviceToHost, js));
    if (ho->episode && out->episode)
      CU_TRY(cudaMemcpyAsync(ho->episode, out->episode, N * CBEV_EPISODE_FIELDS * sizeof(double), cudaMemcpyDeviceToHost,
                             js));
    CU_TRY(cudaEventRecord(e->ev_copy, js));
    e->host_copy_pending = true;
  }
  CU_TRY(cudaEventRecord(e->ev_judge, js));
  if (cbev_launch_render(e, head, mirror, s)) return CBEV_ERR_CUDA;  // cbev_launch_render says why
  if (prof) {
    cudaEventRecord(pe[2], s);
    e->prof_fused[e->prof_n] = fused;
    e->prof_n += 1;
  }
  if ((rc = debug_sync("k_render", s))) return rc;
  CU_TRY(cudaStreamWaitEvent(s, e->ev_judge, 0));  // join (covers the host copies too)
  if (e->cfg.autoreset == CBEV_AUTORESET_SAME_STEP) {
    // the envs that ended in this call: terminal window out, reset from the pool, reset frames rendered at this head
    cbev_launch_same_step_reset(e, out, head, s);
    if ((rc = debug_sync("k_same_step_reset", s))) return rc;
    if (cbev_launch_render(e, head, mirror, s)) return CBEV_ERR_CUDA;  // cbev_launch_render says why
    if ((rc = debug_sync("k_render (same-step reset frames)", s))) return rc;
  }
  CU_TRY(cudaGetLastError());
  e->head = head;
  e->steps += 1;
  return CBEV_OK;
}

int cbev_step_host_ex(cbev_handle e, const void* actions_host, const cbev_step_out* dev_out, const cbev_host_out* host,
                      void* stream) {
  int rc = check_ready(e, true);
  if (rc) return rc;
  if (!actions_host || !host || !host->reward || !host->terminated || !host->truncated) { cbev_set_error("null host buffer"); return CBEV_ERR_ARG; }
  cudaStream_t s = (cudaStream_t)stream;
  const size_t N = (size_t)e->N;
  const size_t abytes = e->cfg.action_mode == CBEV_ACTION_DISCRETE ? N * 8 : N * 12;
  CU_TRY(cudaMemcpyAsync(e->h_actions_dev, actions_host, abytes, cudaMemcpyHostToDevice, s));
  cbev_step_out out;
  if (dev_out) {
    out = *dev_out;
  } else {
    memset(&out, 0, sizeof(out));
    out.reward = e->h_reward_dev;
    out.terminated = e->h_term_dev;
    out.truncated = e->h_trunc_dev;
  }
  return cbev_step_ex(e, e->h_actions_dev, &out, host, stream);  // `stream` joins the side stream: a synchronize covers the copies
}

int cbev_step_host(cbev_handle e, const void* actions_host, double* reward_host, uint8_t* terminated_host,
                   uint8_t* truncated_host, void* stream) {
  cbev_host_out host;
  memset(&host, 0, sizeof(host));
  host.reward = reward_host;
  host.terminated = terminated_host;
  host.truncated = truncated_host;
  return cbev_step_host_ex(e, actions_host, nullptr, &host, stream);
}

int cbev_set_action_repeat(cbev_handle e, int32_t repeat) {
  if (!e) { cbev_set_error("null handle"); return CBEV_ERR_ARG; }
  if (repeat < 1 || repeat > CBEV_MAX_ACTION_REPEAT) {
    cbev_set_error("repeat must lie in [1, %d], got %d", CBEV_MAX_ACTION_REPEAT, (int)repeat);
    return CBEV_ERR_ARG;
  }
  e->action_repeat = repeat;
  return CBEV_OK;
}

int cbev_invalidate(cbev_handle e) {
  if (!e) { cbev_set_error("null handle"); return CBEV_ERR_ARG; }
  { int rc0 = use_device(e); if (rc0) return rc0; }
  CU_TRY(cudaDeviceSynchronize());
  e->was_reset = false;
  e->pool_epoch += 1;
  return CBEV_OK;
}

int64_t cbev_snapshot_row_bytes(cbev_handle e) { return e ? cbev_snap_layout(e, e->pool.max_retreat).row_bytes : -1; }

// shared checks of cbev_snapshot / cbev_restore: engine ready and reset, n in 1..N, 16-byte aligned rows
static int check_snapshot_args(cbev_handle e, const void* rows_mem, int32_t n, const char* what) {
  int rc = check_ready(e, false);
  if (rc) return rc;
  if (!e->was_reset) { cbev_set_error("%s before the first reset (or after cbev_invalidate): no env state", what); return CBEV_ERR_STATE; }
  if (n < 1 || n > e->N) { cbev_set_error("%s: n must be within 1..%d (num_envs), got %d", what, e->N, n); return CBEV_ERR_ARG; }
  if (((uintptr_t)rows_mem & 15) != 0) { cbev_set_error("%s: snapshot rows must be 16-byte aligned", what); return CBEV_ERR_ARG; }
  return CBEV_OK;
}

int cbev_snapshot(cbev_handle e, const int32_t* env_ids_dev, int32_t n, void* dst_dev, int64_t dst_bytes,
                  cbev_snapshot_info* info_out, void* stream) {
  if (!e) { cbev_set_error("null handle"); return CBEV_ERR_ARG; }
  if (!dst_dev || !info_out) { cbev_set_error("cbev_snapshot: null destination or info"); return CBEV_ERR_ARG; }
  int rc = check_snapshot_args(e, dst_dev, n, "cbev_snapshot");
  if (rc) return rc;
  const int64_t row_bytes = cbev_snap_layout(e, e->pool.max_retreat).row_bytes;
  if (dst_bytes < (int64_t)n * row_bytes) {
    cbev_set_error("cbev_snapshot: destination holds %lld bytes, %d rows need %lld (%lld per row)", (long long)dst_bytes,
                   n, (long long)n * row_bytes, (long long)row_bytes);
    return CBEV_ERR_ARG;
  }
  cbev_launch_snapshot(e, env_ids_dev, n, dst_dev, (cudaStream_t)stream);
  if ((rc = debug_sync("k_snapshot", (cudaStream_t)stream))) return rc;
  CU_TRY(cudaGetLastError());
  memset(info_out, 0, sizeof(*info_out));
  info_out->engine_token = e->token;
  info_out->pool_epoch = e->pool_epoch;
  info_out->retreat_slots = e->pool.max_retreat;
  info_out->row_bytes = row_bytes;
  info_out->n_rows = n;
  return CBEV_OK;
}

int cbev_restore(cbev_handle e, const cbev_snapshot_info* info, const void* src_dev, const int32_t* rows_dev,
                 const int32_t* env_ids_dev, int32_t n, void* stream) {
  if (!e) { cbev_set_error("null handle"); return CBEV_ERR_ARG; }
  if (!info || !src_dev) { cbev_set_error("cbev_restore: null info or source"); return CBEV_ERR_ARG; }
  int rc = check_snapshot_args(e, src_dev, n, "cbev_restore");
  if (rc) return rc;
  if (info->engine_token != e->token) { cbev_set_error("cbev_restore: the rows were taken by another engine"); return CBEV_ERR_ARG; }
  if (info->pool_epoch != e->pool_epoch) {
    cbev_set_error("cbev_restore: the rows were taken under pool epoch %d, the engine is at %d (the pool was invalidated "
                   "or replaced since)", info->pool_epoch, e->pool_epoch);
    return CBEV_ERR_STATE;
  }
  if (info->retreat_slots < 0 || info->retreat_slots > e->pool.max_retreat) {
    cbev_set_error("cbev_restore: the rows have %d retreat slots, more than the engine's %d", info->retreat_slots,
                   e->pool.max_retreat);
    return CBEV_ERR_ARG;
  }
  const SnapLayout L = cbev_snap_layout(e, info->retreat_slots);
  if (info->row_bytes != L.row_bytes) {
    cbev_set_error("cbev_restore: row_bytes %lld does not match the %lld of this engine at %d retreat slots",
                   (long long)info->row_bytes, (long long)L.row_bytes, info->retreat_slots);
    return CBEV_ERR_ARG;
  }
  if (info->n_rows < 1 || (!rows_dev && n > info->n_rows)) {
    cbev_set_error("cbev_restore: n = %d with identity rows needs as many rows, the snapshot has %d", n, info->n_rows);
    return CBEV_ERR_ARG;
  }
  cbev_launch_restore(e, L, src_dev, info->n_rows, rows_dev, env_ids_dev, n, (cudaStream_t)stream);
  if ((rc = debug_sync("k_restore", (cudaStream_t)stream))) return rc;
  CU_TRY(cudaGetLastError());
  return CBEV_OK;
}

// Branch state of cbev_lookahead: scene, episode, done + every state section, at least `rows` rows at the pool's
// retreat slots.
static int ensure_branch_state(cbev_engine* e, int32_t rows) {
  const int32_t R = e->pool.max_retreat > 0 ? e->pool.max_retreat : 1;
  if (e->branch.scene && rows <= e->branch_rows && R <= e->branch_retreat) return CBEV_OK;
  CU_TRY(cudaDeviceSynchronize());  // earlier lookahead launches may still read and write the rows being replaced
  rows = std::max(rows, e->branch_rows);
  free_state(e->branch);
  e->branch_rows = e->branch_retreat = 0;
  const int32_t A = e->cfg.max_actors > 0 ? e->cfg.max_actors : 1;
  const StateSections S = cbev_state_sections(e->branch, A, R);
  int rc = dev_alloc(&e->branch.scene, (size_t)rows);
  rc |= dev_alloc(&e->branch.episode, (size_t)rows);
  rc |= dev_alloc(&e->branch.done, (size_t)rows);
  for (int k = 0; k < CBEV_STATE_SECTIONS && !rc; ++k)
    rc |= dev_alloc((uint8_t**)S.field[k], (size_t)rows * S.count[k] * S.esize[k]);
  if (rc) {
    free_state(e->branch);
    return rc;
  }
  e->branch_rows = rows;
  e->branch_retreat = R;
  return CBEV_OK;
}

// Branch render state of cbev_lookahead_obs: staging and render positions for at least `rows` branches at the current
// max_rects (the draw-list stride, which a pool upload may raise).
static int ensure_branch_render(cbev_engine* e, int32_t rows) {
  if (e->br_desc && rows <= e->br_rows && e->br_max_rects == e->max_rects) return CBEV_OK;
  CU_TRY(cudaDeviceSynchronize());  // earlier lookahead and raster launches may still use the buffers being replaced
  rows = std::max(rows, e->br_rows);
  dev_free(e->br_stage_desc); dev_free(e->br_stage_rects); dev_free(e->br_desc); dev_free(e->br_rects);
  e->br_rows = e->br_max_rects = 0;
  const size_t slots = (size_t)rows * e->cfg.frame_stack, rw = (size_t)e->max_rects * CBEV_RECT_WORDS;
  int rc = dev_alloc(&e->br_stage_desc, slots * CBEV_DESC_WORDS);
  rc |= dev_alloc(&e->br_stage_rects, slots * rw);
  rc |= dev_alloc(&e->br_desc, slots * CBEV_DESC_WORDS);
  rc |= dev_alloc(&e->br_rects, slots * rw);
  if (rc) {
    dev_free(e->br_stage_desc); dev_free(e->br_stage_rects); dev_free(e->br_desc); dev_free(e->br_rects);
    return rc;
  }
  e->br_rows = rows;
  e->br_max_rects = e->max_rects;
  return CBEV_OK;
}

// Leaf windows of cbev_lookahead_ex's leaf rows when the caller does not ask for them: room for `bytes`.
static int ensure_branch_window(cbev_engine* e, int64_t bytes) {
  if (e->br_window && bytes <= e->br_window_bytes) return CBEV_OK;
  CU_TRY(cudaDeviceSynchronize());  // earlier raster and row-writer launches may still use the buffer being replaced
  dev_free(e->br_window);
  e->br_window_bytes = 0;
  int rc = dev_alloc(&e->br_window, (size_t)bytes);
  if (rc) return rc;
  e->br_window_bytes = bytes;
  return CBEV_OK;
}

// host checks shared by the lookahead calls (`what` names the entry point in the messages); identity roots start
// from env b unless the call has another root source (`live_roots` false), which checks its own bound
static int check_lookahead_args(cbev_handle e, const int32_t* root_env_ids_dev, int32_t n_branches, int32_t horizon,
                                const void* actions_dev, double gamma, const cbev_lookahead_out* out,
                                const char* what, bool live_roots = true) {
  if (!actions_dev || !out || !out->ret) { cbev_set_error("%s: actions_dev and out->ret are required", what); return CBEV_ERR_ARG; }
  if (n_branches < 1) { cbev_set_error("%s: n_branches must be >= 1, got %d", what, n_branches); return CBEV_ERR_ARG; }
  if (horizon < 1) { cbev_set_error("%s: horizon must be >= 1, got %d", what, horizon); return CBEV_ERR_ARG; }
  if (!std::isfinite(gamma)) { cbev_set_error("%s: gamma must be finite, got %g", what, gamma); return CBEV_ERR_ARG; }
  if (live_roots && !root_env_ids_dev && n_branches > e->N) {
    cbev_set_error("%s: with NULL roots branch b starts from env b, so n_branches must be <= %d (num_envs), got %d", what,
                   e->N, n_branches);
    return CBEV_ERR_ARG;
  }
  return CBEV_OK;
}

int cbev_lookahead(cbev_handle e, const int32_t* root_env_ids_dev, int32_t n_branches, int32_t horizon,
                   const void* actions_dev, double gamma, const cbev_lookahead_out* out, void* stream) {
  if (!e) { cbev_set_error("null handle"); return CBEV_ERR_ARG; }
  int rc = check_lookahead_args(e, root_env_ids_dev, n_branches, horizon, actions_dev, gamma, out, "cbev_lookahead");
  if (rc) return rc;
  if ((rc = check_ready(e, false))) return rc;
  if (!e->was_reset) { cbev_set_error("cbev_lookahead before the first reset (or after cbev_invalidate): no env state"); return CBEV_ERR_STATE; }
  if ((rc = ensure_branch_state(e, n_branches))) return rc;
  cbev_launch_lookahead(e, root_env_ids_dev, n_branches, horizon, actions_dev, gamma, out, false, nullptr, false, 1,
                        (cudaStream_t)stream);
  if ((rc = debug_sync("k_lookahead", (cudaStream_t)stream))) return rc;
  CU_TRY(cudaGetLastError());
  return CBEV_OK;
}

int cbev_lookahead_obs(cbev_handle e, const int32_t* root_env_ids_dev, int32_t n_branches, int32_t horizon,
                       const void* actions_dev, double gamma, const cbev_lookahead_out* out, void* obs_dev,
                       int64_t obs_bytes, void* stream) {
  if (!e) { cbev_set_error("null handle"); return CBEV_ERR_ARG; }
  const char* what = "cbev_lookahead_obs";
  int rc = check_lookahead_args(e, root_env_ids_dev, n_branches, horizon, actions_dev, gamma, out, what);
  if (rc) return rc;
  if (!out->steps) { cbev_set_error("%s: out->steps is required (the leaf-window copy reads it)", what); return CBEV_ERR_ARG; }
  if (!obs_dev) { cbev_set_error("%s: obs_dev is required", what); return CBEV_ERR_ARG; }
  if (((uintptr_t)obs_dev & 15) != 0) { cbev_set_error("%s: obs_dev must be 16-byte aligned", what); return CBEV_ERR_ARG; }
  const int64_t need = (int64_t)n_branches * e->cfg.frame_stack * e->frame_bytes;
  if (obs_bytes < need) {
    cbev_set_error("%s: obs_dev holds %lld bytes, %d leaf windows of %d frames need %lld", what, (long long)obs_bytes,
                   n_branches, e->cfg.frame_stack, (long long)need);
    return CBEV_ERR_ARG;
  }
  if (!e->ring) { cbev_set_error("%s: no observation ring bound (cbev_bind_obs_ring)", what); return CBEV_ERR_STATE; }
  if ((rc = check_ready(e, false))) return rc;
  if (!e->was_reset) { cbev_set_error("%s before the first reset (or after cbev_invalidate): no env state", what); return CBEV_ERR_STATE; }
  if ((rc = ensure_branch_state(e, n_branches))) return rc;
  if ((rc = ensure_branch_render(e, n_branches))) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  // three launches, in stream order: the branches (recording the leaf windows' draw lists), the raster kernel over the
  // recorded positions, the positions that come from the roots' windows (reads out->steps)
  cbev_launch_lookahead(e, root_env_ids_dev, n_branches, horizon, actions_dev, gamma, out, true, nullptr, false, 1, s);
  if ((rc = debug_sync("k_lookahead_obs", s))) return rc;
  if (cbev_launch_render_branches(e, n_branches * e->cfg.frame_stack, obs_dev, s)) return CBEV_ERR_CUDA;  // says why
  if ((rc = debug_sync("k_render (leaf windows)", s))) return rc;
  cbev_launch_leaf_window(e, root_env_ids_dev, n_branches, out->steps, obs_dev, nullptr, s);
  if ((rc = debug_sync("k_leaf_window", s))) return rc;
  CU_TRY(cudaGetLastError());
  return CBEV_OK;
}

// cbev_lookahead_ex and cbev_lookahead_repeat (`what`): the same checks and launches, `repeat` sub-steps per action row
static int lookahead_io(cbev_handle e, const cbev_lookahead_io* io, int32_t n_branches, int32_t horizon,
                        int32_t repeat, const void* actions_dev, double gamma, const cbev_lookahead_out* out,
                        void* stream, const char* what) {
  if (!e) { cbev_set_error("null handle"); return CBEV_ERR_ARG; }
  if (repeat < 1 || repeat > CBEV_MAX_ACTION_REPEAT) {
    cbev_set_error("%s: repeat must lie in [1, %d], got %d", what, CBEV_MAX_ACTION_REPEAT, (int)repeat);
    return CBEV_ERR_ARG;
  }
  if (!io) { cbev_set_error("%s: io is required", what); return CBEV_ERR_ARG; }
  const cbev_snapshot_info* si = io->src_info;
  int rc = check_lookahead_args(e, io->roots, n_branches, horizon, actions_dev, gamma, out, what, si == nullptr);
  if (rc) return rc;
  RowSource src = {};
  if (si) {
    if (!io->src_rows) { cbev_set_error("%s: src_rows is required with src_info", what); return CBEV_ERR_ARG; }
    if (((uintptr_t)io->src_rows & 15) != 0) { cbev_set_error("%s: src_rows must be 16-byte aligned", what); return CBEV_ERR_ARG; }
    if (si->engine_token != e->token) { cbev_set_error("%s: the src rows were taken by another engine", what); return CBEV_ERR_STATE; }
    if (si->pool_epoch != e->pool_epoch) {
      cbev_set_error("%s: the src rows were taken under pool epoch %d, the engine is at %d (the pool was invalidated "
                     "or replaced since)", what, si->pool_epoch, e->pool_epoch);
      return CBEV_ERR_STATE;
    }
    if (si->retreat_slots < 0 || si->retreat_slots > e->pool.max_retreat) {
      cbev_set_error("%s: the src rows have %d retreat slots, more than the engine's %d", what, si->retreat_slots,
                     e->pool.max_retreat);
      return CBEV_ERR_ARG;
    }
    src.L = cbev_snap_layout(e, si->retreat_slots);
    if (si->row_bytes != src.L.row_bytes) {
      cbev_set_error("%s: src row_bytes %lld does not match the %lld of this engine at %d retreat slots", what,
                     (long long)si->row_bytes, (long long)src.L.row_bytes, si->retreat_slots);
      return CBEV_ERR_ARG;
    }
    if (si->n_rows < 1 || (!io->roots && n_branches > si->n_rows)) {
      cbev_set_error("%s: with NULL roots branch b starts from row b, so n_branches must be <= %d (src n_rows), got %d",
                     what, si->n_rows, n_branches);
      return CBEV_ERR_ARG;
    }
    src.rows = io->src_rows;
    src.n_rows = si->n_rows;
  }
  const int64_t win_bytes = (int64_t)n_branches * e->cfg.frame_stack * e->frame_bytes;
  if (io->obs) {
    if (((uintptr_t)io->obs & 15) != 0) { cbev_set_error("%s: obs must be 16-byte aligned", what); return CBEV_ERR_ARG; }
    if (io->obs_bytes < win_bytes) {
      cbev_set_error("%s: obs holds %lld bytes, %d leaf windows of %d frames need %lld", what,
                     (long long)io->obs_bytes, n_branches, e->cfg.frame_stack, (long long)win_bytes);
      return CBEV_ERR_ARG;
    }
  }
  const int64_t row_bytes = cbev_snap_layout(e, e->pool.max_retreat).row_bytes;
  if (io->leaf_rows) {
    if (!io->leaf_info) { cbev_set_error("%s: leaf_info is required with leaf_rows", what); return CBEV_ERR_ARG; }
    if (((uintptr_t)io->leaf_rows & 15) != 0) { cbev_set_error("%s: leaf_rows must be 16-byte aligned", what); return CBEV_ERR_ARG; }
    if (io->leaf_bytes < (int64_t)n_branches * row_bytes) {
      cbev_set_error("%s: leaf_rows holds %lld bytes, %d leaf rows need %lld (%lld per row)", what,
                     (long long)io->leaf_bytes, n_branches, (long long)n_branches * row_bytes, (long long)row_bytes);
      return CBEV_ERR_ARG;
    }
  }
  const bool frames = io->obs || io->leaf_rows;
  if (frames && !out->steps) { cbev_set_error("%s: out->steps is required with obs or leaf_rows (the window copy reads it)", what); return CBEV_ERR_ARG; }
  if (frames && !e->ring) { cbev_set_error("%s: no observation ring bound (cbev_bind_obs_ring)", what); return CBEV_ERR_STATE; }
  if ((rc = check_ready(e, false))) return rc;
  if (!e->was_reset) { cbev_set_error("%s before the first reset (or after cbev_invalidate): no env state", what); return CBEV_ERR_STATE; }
  if ((rc = ensure_branch_state(e, n_branches))) return rc;
  if (frames && (rc = ensure_branch_render(e, n_branches))) return rc;
  if (io->leaf_rows && !io->obs && (rc = ensure_branch_window(e, win_bytes))) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const RowSource* sp = si ? &src : nullptr;
  void* win = io->obs ? io->obs : (io->leaf_rows ? (void*)e->br_window : nullptr);
  // in stream order: the branches; with frames the raster kernel over the recorded leaf positions and the root frames
  // (reads out->steps); with leaf rows the row writer, after every read of the root rows (so they may be overwritten)
  cbev_launch_lookahead(e, io->roots, n_branches, horizon, actions_dev, gamma, out, frames, sp, io->leaf_rows != nullptr,
                        repeat, s);
  if ((rc = debug_sync(repeat > 1 ? "k_lookahead_rep" : "k_lookahead_ex", s))) return rc;
  if (frames) {
    if (cbev_launch_render_branches(e, n_branches * e->cfg.frame_stack, win, s)) return CBEV_ERR_CUDA;  // says why
    if ((rc = debug_sync("k_render (leaf windows)", s))) return rc;
    cbev_launch_leaf_window(e, io->roots, n_branches, out->steps, win, sp, s);
    if ((rc = debug_sync("k_leaf_window", s))) return rc;
  }
  if (io->leaf_rows) {
    cbev_launch_leaf_rows(e, n_branches, win, io->leaf_rows, s);
    if ((rc = debug_sync("k_leaf_rows", s))) return rc;
  }
  CU_TRY(cudaGetLastError());
  if (io->leaf_rows) {  // written last: leaf_info may be the caller's src_info
    cbev_snapshot_info* li = io->leaf_info;
    memset(li, 0, sizeof(*li));
    li->engine_token = e->token;
    li->pool_epoch = e->pool_epoch;
    li->retreat_slots = e->pool.max_retreat;
    li->row_bytes = row_bytes;
    li->n_rows = n_branches;
  }
  return CBEV_OK;
}

int cbev_lookahead_ex(cbev_handle e, const cbev_lookahead_io* io, int32_t n_branches, int32_t horizon,
                      const void* actions_dev, double gamma, const cbev_lookahead_out* out, void* stream) {
  return lookahead_io(e, io, n_branches, horizon, 1, actions_dev, gamma, out, stream, "cbev_lookahead_ex");
}

int cbev_lookahead_repeat(cbev_handle e, const cbev_lookahead_io* io, int32_t n_branches, int32_t horizon,
                          int32_t repeat, const void* actions_dev, double gamma, const cbev_lookahead_out* out,
                          void* stream) {
  return lookahead_io(e, io, n_branches, horizon, repeat, actions_dev, gamma, out, stream, "cbev_lookahead_repeat");
}

int cbev_wait_host_outputs(cbev_handle e) {
  if (!e) { cbev_set_error("null handle"); return CBEV_ERR_ARG; }
  { int rc0 = use_device(e); if (rc0) return rc0; }
  if (!e->host_copy_pending) return CBEV_OK;
  CU_TRY(cudaEventSynchronize(e->ev_copy));
  e->host_copy_pending = false;
  return CBEV_OK;
}

int cbev_upload_fov_mask(cbev_handle e, const uint8_t* mask_host) {
  if (!e) { cbev_set_error("null handle"); return CBEV_ERR_ARG; }
  { int rc0 = use_device(e); if (rc0) return rc0; }
  CU_TRY(cudaDeviceSynchronize());
  dev_free(e->fov_mask);
  if (!mask_host) return CBEV_OK;
  const size_t n = (size_t)e->cfg.fov_size * e->cfg.fov_size;
  std::vector<uint8_t> m(n);
  for (size_t i = 0; i < n; ++i) m[i] = mask_host[i] ? 0xff : 0x00;
  return dev_upload(&e->fov_mask, m.data(), n);
}

// shared checks of cbev_fuse / cbev_fuse_windows: fusion mode, semantic masks, frame_stack >= 3
static int check_fuse_mode(cbev_handle e, int32_t mode) {
  if (mode != CBEV_FUSE_VEHICLE_TEMPORAL && mode != CBEV_FUSE_VEHICLE_WEIGHTED) { cbev_set_error("bad fusion mode %d", mode); return CBEV_ERR_ARG; }
  if (e->cfg.obs_mode != CBEV_OBS_SEMANTIC && e->cfg.obs_mode != CBEV_OBS_SEMANTIC_U8) { cbev_set_error("temporal_fusion_mode requires obs_mode='bev_semantic'"); return CBEV_ERR_ARG; }
  if (e->cfg.frame_stack < 3) { cbev_set_error("temporal_fusion_mode requires frame_stack >= 3"); return CBEV_ERR_ARG; }
  return CBEV_OK;
}

int cbev_fuse(cbev_handle e, int32_t mode, void* out_dev, void* stream) {
  int rc = check_ready(e, true);
  if (rc) return rc;
  if (!out_dev) { cbev_set_error("null output"); return CBEV_ERR_ARG; }
  if ((rc = check_fuse_mode(e, mode))) return rc;
  if (cbev_launch_fuse(e, mode, e->ring, e->N, e->cfg.ring_slots, e->head, out_dev, (cudaStream_t)stream)) {
    cbev_set_error("temporal_fusion_mode requires a semantic_mask_ch with a vehicle channel");
    return CBEV_ERR_ARG;
  }
  CU_TRY(cudaGetLastError());
  return CBEV_OK;
}

int cbev_fuse_windows(cbev_handle e, int32_t mode, const void* windows_dev, int32_t n, void* out_dev, void* stream) {
  if (!e) { cbev_set_error("null handle"); return CBEV_ERR_ARG; }
  if (!windows_dev || !out_dev) { cbev_set_error("cbev_fuse_windows: null windows or output"); return CBEV_ERR_ARG; }
  if ((((uintptr_t)windows_dev | (uintptr_t)out_dev) & 15) != 0) { cbev_set_error("cbev_fuse_windows: windows and output must be 16-byte aligned"); return CBEV_ERR_ARG; }
  if (n < 1) { cbev_set_error("cbev_fuse_windows: n must be >= 1, got %d", n); return CBEV_ERR_ARG; }
  int rc = check_fuse_mode(e, mode);
  if (rc) return rc;
  { int rc0 = use_device(e); if (rc0) return rc0; }
  const int F = e->cfg.frame_stack;
  if (cbev_launch_fuse(e, mode, windows_dev, n, F, F - 1, out_dev, (cudaStream_t)stream)) {
    cbev_set_error("temporal_fusion_mode requires a semantic_mask_ch with a vehicle channel");
    return CBEV_ERR_ARG;
  }
  CU_TRY(cudaGetLastError());
  return CBEV_OK;
}

int cbev_obs_head(cbev_handle e, int32_t* head) {
  if (!e || !head) { cbev_set_error("null argument"); return CBEV_ERR_ARG; }
  *head = e->head;
  return CBEV_OK;
}

int cbev_get_state(cbev_handle e, double* ego_host, double* actors_host) {
  if (!e) { cbev_set_error("null handle"); return CBEV_ERR_ARG; }
  { int rc0 = use_device(e); if (rc0) return rc0; }
  CU_TRY(cudaDeviceSynchronize());
  const size_t N = (size_t)e->N, A = (size_t)(e->cfg.max_actors > 0 ? e->cfg.max_actors : 1);
  if (ego_host) {
    std::vector<double> eg(N * 24);
    std::vector<int32_t> ei(N * 8);
    std::vector<unsigned long long> tv(N * CBEV_TGT_WORDS);
    CU_TRY(cudaMemcpy(eg.data(), e->st.ego, N * 24 * 8, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(ei.data(), e->st.egoi, N * 8 * 4, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(tv.data(), e->st.tgt_vis, N * CBEV_TGT_WORDS * 8, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < N; ++i) {
      double* o = ego_host + i * 16;
      for (int k = 0; k < 9; ++k) o[k] = eg[i * 24 + k];  // x,y,yaw,v,x1,y1,yaw1,v1,acc
      o[9] = (double)ei[i * 8 + 0];                        // tidx
      o[10] = eg[i * 24 + 9];                              // t
      o[11] = eg[i * 24 + 10];                             // dist2goal
      o[12] = eg[i * 24 + 11];                             // dist2goal_1
      o[13] = eg[i * 24 + 12];                             // s_prev
      o[14] = (double)(uint32_t)(tv[i * CBEV_TGT_WORDS] & 0xffffffffull);  // first 64 targets
      o[15] = (double)(uint32_t)(tv[i * CBEV_TGT_WORDS] >> 32);
    }
  }
  if (actors_host) {
    std::vector<double> x(N * A), y(N * A), yaw(N * A), v(N * A), tm(N * A);
    std::vector<int32_t> ti(N * A);
    std::vector<uint8_t> fl(N * A);
    CU_TRY(cudaMemcpy(x.data(), e->st.ax, N * A * 8, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(y.data(), e->st.ay, N * A * 8, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(yaw.data(), e->st.ayaw, N * A * 8, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(v.data(), e->st.av, N * A * 8, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(tm.data(), e->st.atarget_mps, N * A * 8, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(ti.data(), e->st.atidx, N * A * 4, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(fl.data(), e->st.aflags, N * A, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < N * A; ++i) {
      double* o = actors_host + i * 8;
      o[0] = x[i]; o[1] = y[i]; o[2] = yaw[i]; o[3] = v[i]; o[4] = (double)ti[i]; o[5] = (double)(fl[i] & 15);
      o[6] = tm[i]; o[7] = (double)fl[i];
    }
  }
  return CBEV_OK;
}

int cbev_set_ego_state(cbev_handle e, const double* ego_host) {
  if (!e || !ego_host) { cbev_set_error("null argument"); return CBEV_ERR_ARG; }
  { int rc0 = use_device(e); if (rc0) return rc0; }
  CU_TRY(cudaDeviceSynchronize());
  const size_t N = (size_t)e->N;
  std::vector<double> eg(N * 24);
  std::vector<int32_t> ei(N * 8);
  CU_TRY(cudaMemcpy(eg.data(), e->st.ego, N * 24 * 8, cudaMemcpyDeviceToHost));
  CU_TRY(cudaMemcpy(ei.data(), e->st.egoi, N * 8 * 4, cudaMemcpyDeviceToHost));
  for (size_t i = 0; i < N; ++i) {
    const double* o = ego_host + i * 16;
    for (int k = 0; k < 9; ++k) eg[i * 24 + k] = o[k];
    ei[i * 8 + 0] = (int32_t)o[9];
  }
  CU_TRY(cudaMemcpy(e->st.ego, eg.data(), N * 24 * 8, cudaMemcpyHostToDevice));
  CU_TRY(cudaMemcpy(e->st.egoi, ei.data(), N * 8 * 4, cudaMemcpyHostToDevice));
  return CBEV_OK;
}

int cbev_set_state(cbev_handle e, const double* ego_host, const double* actors_host) {
  if (!e) { cbev_set_error("null handle"); return CBEV_ERR_ARG; }
  { int rc0 = use_device(e); if (rc0) return rc0; }
  if (ego_host) {
    int rc = cbev_set_ego_state(e, ego_host);
    if (rc) return rc;
  }
  if (actors_host) {
    CU_TRY(cudaDeviceSynchronize());
    const size_t N = (size_t)e->N, A = (size_t)(e->cfg.max_actors > 0 ? e->cfg.max_actors : 1);
    std::vector<double> x(N * A), y(N * A), yaw(N * A), v(N * A), tm(N * A);
    std::vector<int32_t> ti(N * A);
    std::vector<uint8_t> fl(N * A);
    for (size_t i = 0; i < N * A; ++i) {
      const double* o = actors_host + i * 8;
      x[i] = o[0]; y[i] = o[1]; yaw[i] = o[2]; v[i] = o[3];
      ti[i] = (int32_t)o[4];
      tm[i] = o[6];
      fl[i] = (uint8_t)(((int)o[7] & ~15) | ((int)o[5] & 15));  // flags byte with the FSM state of column 5
    }
    CU_TRY(cudaMemcpy(e->st.ax, x.data(), N * A * 8, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(e->st.ay, y.data(), N * A * 8, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(e->st.ayaw, yaw.data(), N * A * 8, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(e->st.av, v.data(), N * A * 8, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(e->st.atarget_mps, tm.data(), N * A * 8, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(e->st.atidx, ti.data(), N * A * 4, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(e->st.aflags, fl.data(), N * A, cudaMemcpyHostToDevice));
  }
  return CBEV_OK;
}

int cbev_set_debug_flags(cbev_handle e, int32_t flags) {
  if (!e) { cbev_set_error("null handle"); return CBEV_ERR_ARG; }
  if (flags & ~CBEV_DBG_KNOWN) {
    cbev_set_error("unknown debug flags 0x%x (accepted bits: 1, 2, 4, 32, 128, 256, 512, 1024)",
                   (unsigned)(flags & ~CBEV_DBG_KNOWN));
    return CBEV_ERR_ARG;
  }
  e->debug_flags = flags;
  if ((flags & CBEV_DBG_TRACE) && !e->trace) return dev_alloc(&e->trace, (size_t)e->N * 8);
  return CBEV_OK;
}

int cbev_debug_read_trace(cbev_handle e, uint64_t* host_out) {
  if (!e || !host_out) { cbev_set_error("null argument"); return CBEV_ERR_ARG; }
  { int rc0 = use_device(e); if (rc0) return rc0; }
  if (!e->trace) { cbev_set_error("tracing is off (set debug flag 4 first)"); return CBEV_ERR_STATE; }
  CU_TRY(cudaDeviceSynchronize());
  CU_TRY(cudaMemcpy(host_out, e->trace, (size_t)e->N * 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  return CBEV_OK;
}

int cbev_keep_fov(cbev_handle e, int32_t on) {
  if (!e) { cbev_set_error("null handle"); return CBEV_ERR_ARG; }
  e->keep_fov = on != 0;
  return CBEV_OK;
}

int cbev_copy_fov(cbev_handle e, uint8_t* fov_dev, void* stream) {
  if (!e || !fov_dev) { cbev_set_error("null argument"); return CBEV_ERR_ARG; }
  { int rc0 = use_device(e); if (rc0) return rc0; }
  if (!e->keep_fov) { cbev_set_error("palette frames are not kept: call cbev_keep_fov(h, 1) before stepping"); return CBEV_ERR_STATE; }
  size_t bytes = (size_t)e->N * e->cfg.fov_size * e->cfg.fov_size;
  CU_TRY(cudaMemcpyAsync(fov_dev, e->fov, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return CBEV_OK;
}

int cbev_read_stats(cbev_handle e, double* stats_dev, int32_t reset_after, void* stream) {
  if (!e || !stats_dev) { cbev_set_error("null argument"); return CBEV_ERR_ARG; }
  { int rc0 = use_device(e); if (rc0) return rc0; }
  cudaStream_t s = (cudaStream_t)stream;
  CU_TRY(cudaMemcpyAsync(stats_dev, e->gstats, CBEV_STATS_FIELDS * sizeof(double), cudaMemcpyDeviceToDevice, s));
  double steps = (double)e->steps * (double)e->N;
  CU_TRY(cudaMemcpyAsync(stats_dev + CBEV_S_STEPS, &steps, sizeof(double), cudaMemcpyHostToDevice, s));
  CU_TRY(cudaStreamSynchronize(s));  // `steps` lives on this stack frame
  if (reset_after) {
    CU_TRY(cudaMemsetAsync(e->gstats, 0, CBEV_STATS_FIELDS * sizeof(double), s));
    e->steps = 0;
  }
  return CBEV_OK;
}

int64_t cbev_launch_count(cbev_handle e) { return e ? e->launches : -1; }

int cbev_profile_enable(cbev_handle e, int32_t on) {
  if (!e) { cbev_set_error("null handle"); return CBEV_ERR_ARG; }
  { int rc0 = use_device(e); if (rc0) return rc0; }
  if (on && !e->prof_ev) {
    e->prof_ev = new (std::nothrow) cudaEvent_t[CBEV_PROF_EVENTS * CBEV_PROF_MAX];
    if (!e->prof_ev) return CBEV_ERR_NOMEM;
    for (int i = 0; i < CBEV_PROF_EVENTS * CBEV_PROF_MAX; ++i) CU_TRY(cudaEventCreate(&e->prof_ev[i]));
  }
  e->profiling = on != 0;
  e->prof_n = 0;
  return CBEV_OK;
}

int cbev_profile_read_ex(cbev_handle e, double* move_ms, double* render_ms, double* judge_ms, int64_t* steps) {
  if (!e || !move_ms || !render_ms || !judge_ms || !steps) { cbev_set_error("null argument"); return CBEV_ERR_ARG; }
  { int rc0 = use_device(e); if (rc0) return rc0; }
  double a = 0.0, b = 0.0, c = 0.0;
  if (e->prof_n > 0) CU_TRY(cudaDeviceSynchronize());
  for (int i = 0; i < e->prof_n; ++i) {
    const cudaEvent_t* pe = e->prof_ev + CBEV_PROF_EVENTS * i;
    float t0 = 0.f, t1 = 0.f, t2 = 0.f;
    CU_TRY(cudaEventElapsedTime(&t0, pe[0], pe[1]));
    CU_TRY(cudaEventElapsedTime(&t1, pe[1], pe[2]));
    if (!e->prof_fused[i]) CU_TRY(cudaEventElapsedTime(&t2, pe[3], pe[4]));  // k_step_repeat judges inline: 0
    a += t0;
    b += t1;
    c += t2;
  }
  *move_ms = a;
  *render_ms = b;
  *judge_ms = c;
  *steps = e->prof_n;
  e->prof_n = 0;
  return CBEV_OK;
}

int cbev_profile_read(cbev_handle e, double* sim_ms, double* render_ms, int64_t* steps) {
  double judge = 0.0;
  return cbev_profile_read_ex(e, sim_ms, render_ms, &judge, steps);
}

int cbev_abi_sizes(int32_t* config_bytes, int32_t* pool_desc_bytes, int32_t* step_out_bytes) {
  if (config_bytes) *config_bytes = (int32_t)sizeof(cbev_config);
  if (pool_desc_bytes) *pool_desc_bytes = (int32_t)sizeof(cbev_pool_desc);
  if (step_out_bytes) *step_out_bytes = (int32_t)sizeof(cbev_step_out);
  return CBEV_OK;
}

}  // extern "C"

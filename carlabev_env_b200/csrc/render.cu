// render.cu -- BEV rasteriser + observation writer (one CTA per environment).
//
// Restates, for the GPU, the reference's per-step image path:
//   Scene._scene_step map blit + ActorManager.draw_all (src/scenes/scene.py:93-95,
//   src/managers/actor_manager.py:121-132) -> FovRenderer crop / pygame.transform.rotate /
//   compose (envs/fov.py:70-94, envs/world.py:137-157) -> Hero.draw (src/actors/hero.py:26-32)
//   -> CarlaBEV.render (envs/carlabev.py:233-236) -> ResizeObservation (cv2 INTER_AREA 128->96)
//   -> SemanticMaskWrapper / GrayscaleObservation -> FrameStackObservation
//   (envs/__init__.py:62-83, wrappers/rgb_to_semantic.py:65-142).
//
// Pipeline inside one CTA (all on-chip between the map read and the observation write):
//   1. TMA 2-D tile load of the class-map crop (16-byte aligned superset) into shared memory.  Out-of-map texels are
//      zero-filled by the TMA unit = class 0 = NON_DRIVABLE, which is exactly the padded render
//      surface of the reference (envs/world.py:80-87), so no padded copy of the map exists.
//   2. the sim kernel's clipped draw list is painted over the tile in draw order.
//   3. every FOV pixel is inverse-mapped through pygame's 16.16 fixed-point rotate walk
//      (or the exact 90-degree permutation) into the tile -> 128x128 palette-index image.
//   4. 2x2 area taps (weights in 1/16, round-half-even == cv2 INTER_AREA for 128->96) and exact
//      colour equality give one channel bitmask per 96x96 pixel.
//   5. masks are expanded to float32 planes (or 0 / 1 byte planes, CBEV_OBS_SEMANTIC_U8) and streamed to HBM with
//      coalesced 16-byte stores, once per ring slot the frame belongs to.
#include <cuda.h>
#include <stdlib.h>

#include <type_traits>

#include "engine.h"

namespace {

constexpr int RT = 256;  // threads per CTA

__constant__ uint32_t c_pal_rg[CBEV_PAL_COUNT];   // R | G << 16
__constant__ uint32_t c_pal_b[CBEV_PAL_COUNT];
__constant__ uint32_t c_pal_key[CBEV_PAL_COUNT];  // R | G << 8 | B << 16
__constant__ uint8_t c_chan_mask[6][CBEV_PAL_COUNT + 1];  // [mask mode][palette index or NONE] -> channel bits

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* tmap, int x, int y, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(tmap), "r"(smem_u32(bar)), "r"(x), "r"(y)
      : "memory");
}
__device__ __forceinline__ void st_f4(float* p, float a, float b, float c, float d) {
  asm volatile("st.global.cs.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
// 1.0f (0x3f800000) if bit `pos` of m is set, else 0.0f: sign-extending 1-bit field extract, then one AND
__device__ __forceinline__ uint32_t bit_to_f32(uint32_t m, int pos) {
  int32_t s;
  asm("bfe.s32 %0, %1, %2, 1;" : "=r"(s) : "r"(m), "r"(pos));
  return (uint32_t)s & 0x3f800000u;
}
__device__ __forceinline__ void st_b4(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.global.cs.v4.b32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void st_u4(void* p, uint4 v) {
  asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}

struct RenderParams {
  int32_t N, fov, crop, anchor_x, anchor_y;
  int32_t frame_stack, ring_slots, head, mirror;  // mirror = slot offset (L - F + 1)
  int64_t frame_bytes;
  int32_t generic_rotate;  // take the generic (range-tested) rotate path even where the window corners prove it unneeded
  int32_t blk83;  // k_render_any: the 8:3 block shortcut is on (separate output bytes + block flags behind the tables)
  int32_t list_cap;  // k_render_any: entries of the mixed-output work list; the resize runs in bands of that many outputs
  const int32_t* desc;
  const uint32_t* rects;
  const int32_t* order;       // CTA -> env (heavy envs first), or null
  int32_t* order_cnt;         // zeroed here for the next step's k_move
  int32_t max_rects;
  uint8_t* fov_out;  // [N][S][S] palette-index frames (nullable)
  const uint8_t* fov_mask;  // [S][S] 0x00 / 0xff or null (fov_masked)
  void* ring;
  int32_t obs_h, obs_w, rs_mode, rs_words;  // rs_mode: CBEV_RS_* (engine.h); rs_words = size of rs_tab
  const int32_t* rs_tab;                    // cv2 area tables of both axes (api.cu: build_resize_tables)
  unsigned long long* trace;                // [N][8] phase timestamps or null (cbev_debug_read_trace)
  int32_t hero_w;                           // ego square (hero.py:17), 4 px at size 128
  int32_t nbx, nby, box_h, region_bytes;    // k_render_any: strips x row boxes of the fetch window; tile / output region
};

__device__ __forceinline__ void trace_mark(const RenderParams& P, int env, int slot) {
  if (P.trace != nullptr && threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    P.trace[(size_t)env * 8 + slot] = t;
    if (slot == 0) {
      unsigned sm;
      asm volatile("mov.u32 %0, %%smid;" : "=r"(sm));
      P.trace[(size_t)env * 8 + 6] = sm;
    }
  }
}

// cv2 INTER_AREA 128 -> 96: dst pixel d covers src taps s0 = floor(4d/3), s0+1 with weights
// (3-ph, 1+ph)/4, ph = d % 3 (SURVEY.md A.7).  Product weights are in 1/16 units; sums are exact.
__device__ __forceinline__ uint32_t round_half_even_16(uint32_t s) {
  uint32_t q = s >> 4, r = s & 15u;
  return q + ((r > 8u) || (r == 8u && (q & 1u)));
}

// resolve the resized pixel: returns palette index (exact colour equality) or CBEV_PAL_COUNT (no class)
__device__ __forceinline__ uint32_t blend_rgb(uint32_t c00, uint32_t c01, uint32_t c10, uint32_t c11, uint32_t wx0,
                                              uint32_t wx1, uint32_t wy0, uint32_t wy1, const uint32_t* s_rg,
                                              const uint32_t* s_b) {
  uint32_t rg = wy0 * (wx0 * s_rg[c00] + wx1 * s_rg[c01]) + wy1 * (wx0 * s_rg[c10] + wx1 * s_rg[c11]);
  uint32_t b = wy0 * (wx0 * s_b[c00] + wx1 * s_b[c01]) + wy1 * (wx0 * s_b[c10] + wx1 * s_b[c11]);
  uint32_t R = round_half_even_16(rg & 0xffffu), G = round_half_even_16(rg >> 16), B = round_half_even_16(b);
  return R | (G << 8) | (B << 16);
}

// one output byte of the 96x96 image from its 2x2 taps: channel bitmask (semantic) or gray level
template <int OBS_MODE>
__device__ __forceinline__ uint32_t resolve_px(uint32_t c00, uint32_t c01, uint32_t c10, uint32_t c11, uint32_t wx0,
                                               uint32_t wx1, uint32_t wy0, uint32_t wy1, const uint32_t* s_rg,
                                               const uint32_t* s_b, const uint32_t* s_key, const uint8_t* s_cm) {
  const bool same = c00 == c01 && c00 == c10 && c00 == c11;
  if (OBS_MODE == CBEV_OBS_SEMANTIC) {
    uint32_t cls = c00;
    if (!same) {
      const uint32_t key = blend_rgb(c00, c01, c10, c11, wx0, wx1, wy0, wy1, s_rg, s_b);
      cls = CBEV_PAL_COUNT;
#pragma unroll
      for (int q = 0; q < CBEV_PAL_TL_YELLOW; ++q) cls = (key == s_key[q]) ? q : cls;
    }
    return s_cm[cls];
  }
  const uint32_t key = same ? s_key[c00] : blend_rgb(c00, c01, c10, c11, wx0, wx1, wy0, wy1, s_rg, s_b);
  // GrayscaleObservation: sum(rgb * [0.2125, 0.7154, 0.0721]).astype(uint8), float64 left-to-right
  const double g = __dadd_rn(__dadd_rn(__dmul_rn((double)(key & 255u), 0.2125),
                                       __dmul_rn((double)((key >> 8) & 255u), 0.7154)),
                             __dmul_rn((double)(key >> 16), 0.0721));
  return (uint32_t)(int)g & 255u;
}

// exact colour equality of a resized pixel -> channel bitmask (semantic) or gray level (GrayscaleObservation)
template <int OBS_MODE>
__device__ __forceinline__ uint32_t classify_key(uint32_t key, const uint32_t* s_key, const uint8_t* s_cm) {
  if (OBS_MODE == CBEV_OBS_SEMANTIC) {
    uint32_t cls = CBEV_PAL_COUNT;
#pragma unroll
    for (int q = 0; q < CBEV_PAL_TL_YELLOW; ++q) cls = (key == s_key[q]) ? q : cls;
    return s_cm[cls];
  }
  const double g = __dadd_rn(__dadd_rn(__dmul_rn((double)(key & 255u), 0.2125),
                                       __dmul_rn((double)((key >> 8) & 255u), 0.7154)),
                             __dmul_rn((double)(key >> 16), 0.0721));
  return (uint32_t)(int)g & 255u;
}

// CBEV_OBS_SEMANTIC_U8 store phase: 16 mask bytes (bit c = channel c) per thread as one uint4; channel c of them is
// (w >> c) & 0x01010101 on each word, one 16-byte streaming store per channel plane (plane % 16 == 0, api.cu checks)
template <int CHANNELS>
__device__ __forceinline__ void store_u8_planes(uint8_t* base, const uint8_t* s_out, int plane, int tid, int nt) {
  for (int q = tid; q < plane / 16; q += nt) {
    const uint4 m = ((const uint4*)s_out)[q];
#pragma unroll
    for (int c = 0; c < CHANNELS; ++c)
      st_u4(base + (size_t)c * plane + 16 * q,
            make_uint4((m.x >> c) & 0x01010101u, (m.y >> c) & 0x01010101u, (m.z >> c) & 0x01010101u,
                       (m.w >> c) & 0x01010101u));
  }
}

// The 128 x 128 palette-index frame lives in shared memory with its 16-byte chunks XOR-swizzled by the row
// (chunk' = chunk ^ (row & 7)): the rotate writes 8-row x 16-px patches per warp, and with this layout those word
// stores -- like every row-wise 16-byte read of the later phases -- hit 32 different banks.
__device__ __forceinline__ int fov_word(int row, int cw) { return row * 32 + ((((cw >> 2) ^ row) & 7) << 2) + (cw & 3); }
__device__ __forceinline__ int fov_byte(int row, int x) { return row * 128 + ((((x >> 4) ^ row) & 7) << 4) + (x & 15); }

// The EnvConfig.size = 128, obs_size = (96, 96) specialisation (4x4-block two-pass resize) -- every BASELINE
// configuration.  Other view sizes and observation sizes go through k_render_any below.
// U8 (CBEV_OBS_SEMANTIC_U8, with OBS_MODE = CBEV_OBS_SEMANTIC) changes the store phase only: 0 / 1 byte planes.
template <int OBS_MODE, int CHANNELS, bool U8 = false>
__global__ void __launch_bounds__(RT, 4)
k_render(RenderParams P, const __grid_constant__ CUtensorMap tmap, int mask_mode) {
  extern __shared__ __align__(128) uint8_t smem[];
  // layout: [tile: CBEV_TILE_H rows x CBEV_TILE_W | re-used as: 96x96 output bytes + mixed-block worklist / RGB staging
  //          (which runs on into the fov region)] [fov 128x128, swizzled] [tables] [mbar] [draw list]
  constexpr int S = 128;
  constexpr int pitch = CBEV_TILE_W;
  constexpr int tile_bytes = CBEV_TILE_W * CBEV_TILE_H;
  uint8_t* s_tile = smem;
  uint8_t* const s_region = smem;  // start of the tile region (16-byte aligned), re-used after the rotate
  uint8_t* s_fov = smem + tile_bytes;
  uint32_t* s_rg = (uint32_t*)(s_fov + S * S);
  uint32_t* s_b = s_rg + 16;
  uint32_t* s_key = s_b + 16;
  int32_t* s_desc = (int32_t*)(s_key + 16);
  uint64_t* s_bar = (uint64_t*)(s_desc + CBEV_DESC_WORDS);
  uint8_t* s_cm = (uint8_t*)(s_bar + 2);     // channel bits per palette index for this mask mode
  int* s_count = (int*)(s_cm + 16);
  uint32_t* s_rects = (uint32_t*)(s_count + 4);  // draw list (max_rects x 2 words)

  const int env = P.order != nullptr ? P.order[blockIdx.x] : blockIdx.x;
  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;
  if (blockIdx.x == 0 && tid < 2 && P.order_cnt != nullptr) P.order_cnt[tid] = 0;
  const int32_t* d = P.desc + (size_t)env * CBEV_DESC_WORDS;
  const int flags = d[RD_FLAGS];
  if (flags & 2) return;  // masked-out env of a partial reset
  trace_mark(P, env, 0);

  if (tid == 0) {
    mbar_init(s_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    mbar_expect_tx(s_bar, (uint32_t)tile_bytes);
    // the TMA unit needs a 16-byte aligned inner coordinate (measured on B200: an unaligned x raises
    // "illegal instruction"), so fetch the aligned superset [ox & ~15, +CBEV_TILE_W) and index it with +shift
    tma_load_2d(s_tile, &tmap, d[RD_OX] & ~15, d[RD_OY], s_bar);
    *s_count = 0;
  }
  if (tid < CBEV_DESC_WORDS) s_desc[tid] = d[tid];
  if (tid < CBEV_PAL_COUNT) {
    s_rg[tid] = c_pal_rg[tid];
    s_b[tid] = c_pal_b[tid];
    s_key[tid] = c_pal_key[tid];
  }
  if (tid <= CBEV_PAL_COUNT) s_cm[tid] = c_chan_mask[mask_mode][tid];
  // the draw list travels while the tile is in flight: one coalesced load instead of one dependent global
  // load per rectangle after the tile has landed (under the store traffic of the other CTAs each costs ~0.6 us)
  const int nrects = d[RD_NRECTS];
  {
    // speculative: every slot of the list is fetched without waiting for the count (no dependent load)
    const uint32_t* rl = P.rects + (size_t)env * P.max_rects * CBEV_RECT_WORDS;
    for (int r = tid; r < P.max_rects * CBEV_RECT_WORDS; r += RT) s_rects[r] = rl[r];
  }
  __syncthreads();
  mbar_wait(s_bar, 0);
  s_tile += s_desc[RD_OX] & 15;  // fetch-window pixel (x, y) lives at s_tile[y * pitch + x]
  trace_mark(P, env, 1);

  // ---- 2. draw list, in order (later rects overwrite earlier ones) ----
  // Runs of consecutive rects with the same colour (all vehicles, all pedestrians, the route targets) are painted in
  // parallel, one rect per thread: overlapping rects of one run write the same value, so their order does not matter;
  // runs follow each other in list order, which is all "later overwrites earlier" needs.
  if (nrects > 0) {
    int r = 0;
    while (r < nrects) {  // r, e are uniform over the CTA: every warp scans the run boundaries itself
      const uint32_t pal = s_rects[2 * r + 1] >> 24;
      int e = r;
      for (;;) {  // end of the run that starts at r
        const int idx = e + lane;
        const unsigned same = __ballot_sync(0xffffffffu, idx < nrects && (s_rects[2 * idx + 1] >> 24) == pal);
        if (same == 0xffffffffu) { e += 32; continue; }
        e += __ffs(~same) - 1;
        break;
      }
      for (int q = r + tid; q < e; q += RT) {
        const uint32_t w0 = s_rects[2 * q], w1 = s_rects[2 * q + 1];
        const int x0 = w0 & 0xffff, y0 = w0 >> 16, w = (w1 & 0xfff) + 1, h = ((w1 >> 12) & 0xfff) + 1;
        uint8_t* row = s_tile + y0 * pitch + x0;
        for (int yy = 0; yy < h; ++yy, row += pitch)
          for (int xx = 0; xx < w; ++xx) row[xx] = (uint8_t)pal;
      }
      r = e;
      __syncthreads();
    }
    trace_mark(P, env, 7);
  }

  trace_mark(P, env, 2);
  // ---- 3. rotate + compose + ego square -> 128x128 palette-index FOV ----
  // Thread mapping: a warp covers 16-px x 8-row patches (lane = 4 px of one row: lx = lane & 3, ly = lane >> 2).  With
  // the tile pitch an odd number of 16-byte chunks, the 32 byte-gathers of one instruction spread over the banks for
  // every heading (<= 2-way, against up to 28-way for a warp walking one 128-px row: cars mostly drive along the axes,
  // which is exactly the worst case of a row walk).
  {
    const int mode = s_desc[RD_MODE], turns = s_desc[RD_TURNS];
    const int nx = s_desc[RD_NX], ny = s_desc[RD_NY];
    const int isin = s_desc[RD_ISIN], icos = s_desc[RD_ICOS];
    const int rax = s_desc[RD_AX] + s_desc[RD_XD], ray = s_desc[RD_AY] + s_desc[RD_YD], rcy = s_desc[RD_CY];
    const int left = P.anchor_x - (nx >> 1), top = P.anchor_y - (ny >> 1);  // get_rect(center=anchor)
    const int crop = P.crop;
    const int lim = (crop << 16) - 1;
    const uint32_t bg = (uint32_t)s_desc[RD_BG];  // transform.rotate background = source's first pixel
    const int ex0 = P.anchor_x - 2, ey0 = P.anchor_y - 2;
    // crop pixel (sx, sy) = tile0[sy * pitch + sx]
    const uint8_t* tile0 = s_tile - s_desc[RD_FY] * pitch - s_desc[RD_FX];
    const int lx = lane & 3, ly = lane >> 2;
    // The crop is sized so that the 128x128 window normally lies inside the rotated surface and inside the
    // source range of the fixed-point walk.  Both facts are linear in (x, y): checking the four window corners
    // proves them for every pixel, which removes all per-pixel range tests (the generic loop remains for the rest).
    bool fast = left <= 0 && top <= 0 && left + nx >= S && top + ny >= S && !P.generic_rotate;
    if (mode == 1 && fast) {
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int rxp = ((c & 1) ? S - 1 : 0) - left, ryp = ((c & 2) ? S - 1 : 0) - top;
        const int dx = rax + isin * (rcy - ryp) + rxp * icos, dy = ray - icos * (rcy - ryp) + rxp * isin;
        fast = fast && dx >= 0 && dy >= 0 && dx <= lim && dy <= lim;
      }
    }
    uint32_t* fov32 = (uint32_t*)s_fov;
    if (fast && mode == 1) {
      // 16 samples (4 patches) per iteration: all loads are issued before the first store, so the shared-memory
      // latency is paid once per 16 pixels instead of once per 4 (tile and fov may alias for the compiler)
#pragma unroll 1
      for (int i0 = 0; i0 < 16; i0 += 4) {
        uint32_t packed[4];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const int p = warp * 16 + i0 + g;
          const int oy = (p >> 3) * 8 + ly, ox0 = (p & 7) * 16 + lx * 4;
          const int ryp = oy - top, rxp = ox0 - left;
          int dx = rax + isin * (rcy - ryp) + rxp * icos;
          int dy = ray - icos * (rcy - ryp) + rxp * isin;
          uint32_t pk = 0;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            pk |= (uint32_t)tile0[(dy >> 16) * pitch + (dx >> 16)] << (8 * k);
            dx += icos;
            dy += isin;
          }
          packed[g] = pk;
        }
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const int p = warp * 16 + i0 + g;
          fov32[fov_word((p >> 3) * 8 + ly, (p & 7) * 4 + lx)] = packed[g];
        }
      }
    } else if (fast) {
      // exact 90-degree turns (rotate90): src = base + x * step_x + y * step_y
      int base, stepx, stepy;
      if (turns == 0) { base = 0; stepx = 1; stepy = pitch; }
      else if (turns == 1) { base = crop - 1; stepx = pitch; stepy = -1; }
      else if (turns == 2) { base = (crop - 1) * pitch + crop - 1; stepx = -1; stepy = -pitch; }
      else { base = (crop - 1) * pitch; stepx = -pitch; stepy = 1; }
      base += -left * stepx - top * stepy;
#pragma unroll 4
      for (int i = 0; i < 16; ++i) {
        const int p = warp * 16 + i;
        const int oy = (p >> 3) * 8 + ly, ox0 = (p & 7) * 16 + lx * 4;
        const int a = base + ox0 * stepx + oy * stepy;
        fov32[fov_word(oy, ox0 >> 2)] = (uint32_t)tile0[a] | ((uint32_t)tile0[a + stepx] << 8) |
                                         ((uint32_t)tile0[a + 2 * stepx] << 16) | ((uint32_t)tile0[a + 3 * stepx] << 24);
      }
    } else {
      for (int i = 0; i < 16; ++i) {
        const int p = warp * 16 + i;
        const int oy = (p >> 3) * 8 + ly, ox0 = (p & 7) * 16 + lx * 4;
        const int ryp = oy - top;
        const bool row_in = ryp >= 0 && ryp < ny;
        const int bx = rax + isin * (rcy - ryp);
        const int by = ray - icos * (rcy - ryp);
        uint32_t packed = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int rxp = ox0 + k - left;
          uint32_t v = CBEV_PAL_BLACK;
          if (row_in && rxp >= 0 && rxp < nx) {
            if (mode == 0) {
              int sx, sy;
              if (turns == 0) { sx = rxp; sy = ryp; }
              else if (turns == 1) { sx = crop - 1 - ryp; sy = rxp; }
              else if (turns == 2) { sx = crop - 1 - rxp; sy = crop - 1 - ryp; }
              else { sx = ryp; sy = crop - 1 - rxp; }
              v = tile0[sy * pitch + sx];
            } else {
              int dx = bx + rxp * icos, dy = by + rxp * isin;
              if (dx < 0 || dy < 0 || dx > lim || dy > lim) v = bg;
              else v = tile0[(dy >> 16) * pitch + (dx >> 16)];
            }
          }
          packed |= v << (8 * k);
        }
        fov32[fov_word(oy, ox0 >> 2)] = packed;
      }
    }
    __syncthreads();
    // apply_mask (fov.py:96-99): opaque black corner triangles over the composed frame, before the ego is drawn
    if (P.fov_mask != nullptr) {
      for (int u = tid; u < S * S / 4; u += RT) {
        const uint32_t mk = ((const uint32_t*)P.fov_mask)[u];
        uint32_t* px = fov32 + fov_word(u >> 5, u & 31);
        *px = (*px & ~mk) | ((CBEV_PAL_BLACK * 0x01010101u) & mk);
      }
      __syncthreads();
    }
    // Hero.draw: 4x4 black square centred on the anchor (hero.py:26-32), clipped to the surface
    if (tid < 16) {
      const int x = ex0 + (tid & 3), y = ey0 + (tid >> 2);
      if (x >= 0 && x < S && y >= 0 && y < S) s_fov[fov_byte(y, x)] = CBEV_PAL_BLACK;
    }
  }
  __syncthreads();
  trace_mark(P, env, 3);
  if (P.fov_out != nullptr) {
    uint4* dst = (uint4*)(P.fov_out + (size_t)env * S * S);
    for (int u = tid; u < S * S / 16; u += RT) dst[u] = *(const uint4*)(s_fov + fov_byte(u >> 3, (u & 7) << 4));
  }

  // which ring slots receive this frame: the head slot, or every window slot for a reset frame,
  // each mirrored to slot - mirror when that lands in [0, F-2] (keeps the F-window contiguous)
  const int F = P.frame_stack;
  const int first = (flags & 1) ? P.head - F + 1 : P.head;

  if (OBS_MODE == CBEV_OBS_RGB) {
    // raw render(): (S, S, 3) uint8, staged through shared memory for 16-byte coalesced stores.  The staging area
    // (48 KB) starts at the dead tile and runs on into the frame itself, so the frame is pulled into registers first.
    uint32_t f[S * S / 4 / RT];
#pragma unroll
    for (int i = 0; i < S * S / 4 / RT; ++i) {
      const int u = tid + i * RT;
      f[i] = ((const uint32_t*)s_fov)[fov_word(u >> 5, u & 31)];
    }
    __syncthreads();
    uint8_t* s_rgb = s_region;
    // (a PRMT byte-LUT held in registers instead of these shared-memory look-ups was built and measured on B200:
    //  k_render 0.170 ms against 0.151 ms at 8192 envs -- the extra ALU work costs more than the look-ups; removed)
#pragma unroll
    for (int i = 0; i < S * S / 4 / RT; ++i) {  // 4 pixels -> 12 bytes = 3 words
      const int u = tid + i * RT;
      const uint32_t p4 = f[i];
      const uint32_t k0 = s_key[p4 & 255u], k1 = s_key[(p4 >> 8) & 255u], k2 = s_key[(p4 >> 16) & 255u],
                     k3 = s_key[p4 >> 24];
      uint32_t* o = (uint32_t*)s_rgb + 3 * u;
      o[0] = k0 | (k1 << 24);
      o[1] = (k1 >> 8) | (k2 << 16);
      o[2] = (k2 >> 16) | (k3 << 8);
    }
    __syncthreads();
    uint8_t* dst = (uint8_t*)P.ring + (size_t)env * P.ring_slots * P.frame_bytes + (size_t)P.head * P.frame_bytes;
    for (int u = tid; u < S * S * 3 / 16; u += RT) st_u4(dst + 16 * u, ((const uint4*)s_rgb)[u]);
    return;
  }

  constexpr int OH = 96, OW = 96;
  uint8_t* s_out = s_region;                        // OH x OW bytes: channel bitmask (semantic) or gray level
  {
  // ---- 4. area resize 128 -> 96 + colour equality -> one byte per output pixel ----
  // Every 4x4 source block maps to a 3x3 output block (period of the 4/3 scale on both axes).
  // Pass A: a block whose 16 texels are equal resolves to one table lookup for all 9 outputs; the other
  // blocks go to a worklist.  Pass B: the worklist is processed one output pixel per thread (no divergence).
  constexpr int O = 96;
  uint16_t* s_list = (uint16_t*)(s_region + O * O);  // up to 32*32 mixed blocks
  {
    const int br = tid >> 3, j = tid & 7;  // 32 block rows x 8 strips of 4 blocks (RT == 256)
    uint4 R[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) R[i] = *(const uint4*)(s_fov + fov_byte(4 * br + i, 16 * j));
    uint32_t m[4];
    uint32_t mixed = 0;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const uint32_t w0 = (&R[0].x)[b], w1 = (&R[1].x)[b], w2 = (&R[2].x)[b], w3 = (&R[3].x)[b];
      const uint32_t c = w0 & 255u;
      const bool uni = w0 == w1 && w0 == w2 && w0 == w3 && w0 == c * 0x01010101u;
      m[b] = 0;
      if (uni) {
        if (OBS_MODE == CBEV_OBS_SEMANTIC) m[b] = s_cm[c];
        else m[b] = resolve_px<OBS_MODE>(c, c, c, c, 2, 2, 2, 2, s_rg, s_b, s_key, s_cm);
      } else {
        mixed |= 1u << b;
      }
    }
    // 12 output bytes per row: m0 m0 m0 m1 | m1 m1 m2 m2 | m2 m3 m3 m3 (same for the 3 rows of the block row)
    const uint32_t o0 = m[0] | (m[0] << 8) | (m[0] << 16) | (m[1] << 24);
    const uint32_t o1 = m[1] | (m[1] << 8) | (m[2] << 16) | (m[2] << 24);
    const uint32_t o2 = m[2] | (m[3] << 8) | (m[3] << 16) | (m[3] << 24);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      uint32_t* o = (uint32_t*)(s_out + (3 * br + i) * O + 12 * j);
      o[0] = o0; o[1] = o1; o[2] = o2;
    }
    if (mixed) {
      const int n = __popc(mixed);
      int pos = atomicAdd(s_count, n);
#pragma unroll
      for (int b = 0; b < 4; ++b)
        if (mixed & (1u << b)) s_list[pos++] = (uint16_t)(br * 32 + j * 4 + b);
    }
  }
  __syncthreads();
  {
    const int n9 = *s_count * 9;
    for (int idx = tid; idx < n9; idx += RT) {
      const int blk = s_list[idx / 9], px = idx % 9;
      const int i = px / 3, jj = px % 3;
      const int bry = blk >> 5, bcx = blk & 31;
      const uint8_t* src0 = s_fov + fov_byte(4 * bry + i, 4 * bcx + jj);      // the 2x2 taps stay inside one 4-px block
      const uint8_t* src1 = s_fov + fov_byte(4 * bry + i + 1, 4 * bcx + jj);
      const uint32_t res = resolve_px<OBS_MODE>(src0[0], src0[1], src1[0], src1[1], 3 - jj, 1 + jj, 3 - i, 1 + i, s_rg,
                                                s_b, s_key, s_cm);
      s_out[(3 * bry + i) * O + 3 * bcx + jj] = (uint8_t)res;
    }
  }
  __syncthreads();
  }

  // ---- 5. expand + stream out ----
  trace_mark(P, env, 4);
  for (int slot = first; slot <= P.head; ++slot) {
#pragma unroll 1
    for (int rep = 0; rep < 2; ++rep) {
      int sl = slot;
      if (rep == 1) {
        sl = slot - P.mirror;
        if (P.mirror <= 0 || sl < 0) break;
      }
      uint8_t* base = (uint8_t*)P.ring + ((size_t)env * P.ring_slots + sl) * P.frame_bytes;
      if (U8) {
        store_u8_planes<CHANNELS>(base, s_out, OH * OW, tid, RT);
      } else if (OBS_MODE == CBEV_OBS_SEMANTIC) {
        float* fb = (float*)base;
        const int plane = OH * OW;
        // bit c of each of the 4 pixel bytes -> 0.0f / 1.0f in registers: no shared-memory traffic at all in the
        // store loop (the reads of a shared-memory LUT were 57 % of the kernel's shared-load wavefronts, ncu round 2;
        // top stall mio_throttle)
        for (int q = tid; q < plane / 4; q += RT) {
          const uint32_t m4 = ((const uint32_t*)s_out)[q];
#pragma unroll
          for (int c = 0; c < CHANNELS; ++c)
            st_b4(fb + c * plane + 4 * q, bit_to_f32(m4, c), bit_to_f32(m4, c + 8), bit_to_f32(m4, c + 16),
                  bit_to_f32(m4, c + 24));
        }
      } else {
        for (int q = tid; q < OH * OW / 16; q += RT) st_u4(base + 16 * q, ((const uint4*)s_out)[q]);
      }
    }
  }
  trace_mark(P, env, 5);
}

// ---- any view size, any observation size ------------------------------------------------------------------------
// EnvConfig.size in {64, 128, 256} (SURVEY.md section 8 row f4: hero.py:14-17, world.py:38-49; the view, the crop and
// the map scale with it) and any EnvConfig.obs_size.  Same pipeline as k_render without its 128 / 96 specialisations:
//   * the fetch window (<= ceil(S * sqrt 2) + 2 px on a side, 365 px at S = 256) exceeds one TMA box (<= 256 per
//     dimension), so it lands as `nbx` column strips of CBEV_ANY_BOX_W = 128 bytes x `nby` row boxes, all on one
//     mbarrier.  The tensor map uses the 128-byte TMA swizzle (16-byte chunk ^= row & 7): with a dense 128-byte pitch
//     every row would start in bank 0 and a heading along a map axis would put the 32 byte-gathers of an instruction
//     into one bank; swizzled, the 16-px x 8-row warp patches of the rotate are conflict-free or 2-way.
//     Window byte (x, y) lives at ((x >> 7) * tile_h + y) * 128 + (x & 127), XOR (y & 7) << 4;
//   * the frame is stored with a pitch of S + 16 bytes (an odd number of 16-byte chunks: rows rotate through the banks);
//   * cv2.resize(INTER_AREA): copy / 2x2 integer path / float32 area tables when shrinking -- with a shortcut for
//     outputs whose whole source footprint is one colour (the weights sum to 1 within 1e-6, so the result is that
//     colour exactly) -- and OpenCV's 8-bit bilinear kernel on area-mode coefficients when an axis enlarges (64 -> 96).
// One CTA per env: 256 threads (S <= 128), 1024 threads and ~220 KB of shared memory at S = 256 (one CTA per SM).
// U8 as in k_render: the store phase writes 0 / 1 byte planes.
template <int OBS_MODE, int CHANNELS, bool U8 = false>
__global__ void __launch_bounds__(1024, 1)
k_render_any(RenderParams P, const __grid_constant__ CUtensorMap tmap, int mask_mode) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // layout: [tile strips (1024-byte aligned: swizzle period) | re-used as the OH x OW output bytes] [frame S x (S + 16)]
  //         [tables] [mbar] [draw list] [resize tables]
  // (the alignment is declared, not fixed up at run time, so that the tile's address folds into the gathers' LDS)
  uint8_t* const smem = smem_raw;
  if (smem_u32(smem_raw) & 1023u) __trap();
  const int S = P.fov, NT = blockDim.x;
  const int FP = S + 16;  // frame pitch
  constexpr int BW = CBEV_ANY_BOX_W;
  const int tile_h = P.box_h * P.nby;
  const int tile_bytes = BW * P.nbx * tile_h;
  uint8_t* const s_tile = smem;
  uint8_t* const s_fov = smem + P.region_bytes;
  uint32_t* s_rg = (uint32_t*)(s_fov + S * FP);
  uint32_t* s_b = s_rg + 16;
  uint32_t* s_key = s_b + 16;
  int32_t* s_desc = (int32_t*)(s_key + 16);
  uint64_t* s_bar = (uint64_t*)(s_desc + CBEV_DESC_WORDS);
  uint8_t* s_cm = (uint8_t*)(s_bar + 2);
  uint8_t* s_cmu = s_cm + 16;  // palette index -> output byte of a single-colour footprint (= classify_key of its colour)
  float4* s_palf = (float4*)(s_cmu + 16);  // palette index -> (R, G, B) as float32, for the area sums
  uint32_t* s_rects = (uint32_t*)(s_palf + 16);
  int32_t* s_tab = (int32_t*)(s_rects + ((P.max_rects * CBEV_RECT_WORDS + 3) & ~3));
  // 8:3 block shortcut (P.blk83, below): one flag byte per 8 x 8 source block and output bytes of their own, because
  // they are written while the rotate still reads the tile
  uint8_t* s_bflag = (uint8_t*)(s_tab + P.rs_words);
  uint8_t* s_out_sep = s_bflag + ((((S >> 3) * (S >> 3)) + 15) & ~15);

  const int env = P.order != nullptr ? P.order[blockIdx.x] : blockIdx.x;
  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5, nwarps = NT >> 5;
  if (blockIdx.x == 0 && tid < 2 && P.order_cnt != nullptr) P.order_cnt[tid] = 0;
  const int32_t* d = P.desc + (size_t)env * CBEV_DESC_WORDS;
  const int flags = d[RD_FLAGS];
  if (flags & 2) return;  // masked-out env of a partial reset
  trace_mark(P, env, 0);

  if (tid == 0) {
    mbar_init(s_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    mbar_expect_tx(s_bar, (uint32_t)tile_bytes);
    const int x0 = d[RD_OX] & ~15, y0 = d[RD_OY];  // 16-byte aligned inner coordinate (k_render)
    for (int bx = 0; bx < P.nbx; ++bx)
      for (int by = 0; by < P.nby; ++by)
        tma_load_2d(s_tile + (size_t)(bx * tile_h + by * P.box_h) * BW, &tmap, x0 + bx * BW, y0 + by * P.box_h, s_bar);
  }
  if (tid < CBEV_DESC_WORDS) s_desc[tid] = d[tid];
  if (tid < CBEV_PAL_COUNT) {
    s_rg[tid] = c_pal_rg[tid];
    s_b[tid] = c_pal_b[tid];
    s_key[tid] = c_pal_key[tid];
  }
  if (tid <= CBEV_PAL_COUNT) s_cm[tid] = c_chan_mask[mask_mode][tid];
  const int nrects = d[RD_NRECTS];
  {
    const uint32_t* rl = P.rects + (size_t)env * P.max_rects * CBEV_RECT_WORDS;
    for (int r = tid; r < P.max_rects * CBEV_RECT_WORDS; r += NT) s_rects[r] = rl[r];
  }
  for (int u = tid; u < P.rs_words; u += NT) s_tab[u] = P.rs_tab[u];
  __syncthreads();
  if (OBS_MODE != CBEV_OBS_RGB && tid < CBEV_PAL_COUNT) {
    const uint32_t kk = s_key[tid];
    s_cmu[tid] = (uint8_t)classify_key<OBS_MODE>(kk, s_key, s_cm);
    s_palf[tid] = make_float4((float)(kk & 255u), (float)((kk >> 8) & 255u), (float)(kk >> 16), 0.f);
  }
  mbar_wait(s_bar, 0);
  const int shift = s_desc[RD_OX] & 15;
  const int xmax = BW * P.nbx - 1, ymax = tile_h - 1;
  // window pixel (x, y), x already shifted by the alignment slack -> byte offset in the swizzled strips
  auto tile_raw = [&](int x, int y) { return (((x >> 7) * tile_h + y) * BW + (x & (BW - 1))) ^ ((y & 7) << 4); };
  // the same, clamped: a degenerate view can point outside the window
  auto tile_off = [&](int x, int y) { return tile_raw(min(max(x + shift, 0), xmax), min(max(y, 0), ymax)); };
  trace_mark(P, env, 1);

  // ---- 2. draw list, in order: one rect per thread inside a run of equal colour (k_render) ----
  {
    int r = 0;
    while (r < nrects) {
      const uint32_t pal = s_rects[2 * r + 1] >> 24;
      int e = r + 1;
      while (e < nrects && (s_rects[2 * e + 1] >> 24) == pal) ++e;
      for (int q = r + tid; q < e; q += NT) {
        const uint32_t w0 = s_rects[2 * q], w1 = s_rects[2 * q + 1];
        const int x0 = w0 & 0xffff, y0 = w0 >> 16, w = (w1 & 0xfff) + 1, h = ((w1 >> 12) & 0xfff) + 1;
        for (int yy = 0; yy < h; ++yy)
          for (int xx = 0; xx < w; ++xx) s_tile[tile_off(x0 + xx, y0 + yy)] = (uint8_t)pal;
      }
      r = e;
      __syncthreads();
    }
  }
  trace_mark(P, env, 2);

  // ---- 3. rotate + compose + ego square -> S x S palette-index frame (fov.py:84-94, SURVEY.md A.6) ----
  {
    const int mode = s_desc[RD_MODE], turns = s_desc[RD_TURNS];
    const int nx = s_desc[RD_NX], ny = s_desc[RD_NY];
    const int isin = s_desc[RD_ISIN], icos = s_desc[RD_ICOS];
    const int rax = s_desc[RD_AX] + s_desc[RD_XD], ray = s_desc[RD_AY] + s_desc[RD_YD], rcy = s_desc[RD_CY];
    const int left = P.anchor_x - (nx >> 1), top = P.anchor_y - (ny >> 1);  // get_rect(center=anchor)
    const int crop = P.crop;
    const int lim = (crop << 16) - 1;
    const uint32_t bg = (uint32_t)s_desc[RD_BG];
    const int fx = s_desc[RD_FX] - shift, fy = s_desc[RD_FY];  // crop pixel (sx, sy) = window byte (sx - fx, sy - fy)
    // As in k_render: when the four view corners lie inside the rotated surface and inside the source range, every
    // pixel does (both conditions are linear in (x, y)) and the per-pixel range tests and clamps fall away.
    bool fast = left <= 0 && top <= 0 && left + nx >= S && top + ny >= S && !P.generic_rotate && mode == 1;
    if (fast) {
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int rxp = ((c & 1) ? S - 1 : 0) - left, ryp = ((c & 2) ? S - 1 : 0) - top;
        const int dx = rax + isin * (rcy - ryp) + rxp * icos, dy = ray - icos * (rcy - ryp) + rxp * isin;
        fast = fast && dx >= 0 && dy >= 0 && dx <= lim && dy <= lim;
      }
    }
    // a warp covers 16-px x 8-row patches (lane = 4 px of one row), as in k_render
    const int lx = lane & 3, ly = lane >> 2;
    const int pw = S >> 4, pw_log = 31 - __clz(pw);  // patches per row (a power of two)
    const int npatch = pw * (S >> 3);
    // 8:3 block shortcut (S : obs = 8 : 3 on both axes, e.g. 256 -> 96): every 8 x 8 source block is exactly the
    // footprint of a 3 x 3 output block, and a patch is two such blocks.  A block whose 64 texels are one colour gives
    // nine outputs of that colour (the area weights sum to 1 within 1e-6) straight from the rotate's registers: it is
    // never stored to the frame nor visited by the resize.  The other blocks -- and those under the ego square, which
    // is drawn into the frame afterwards -- are flagged and take the table resize below.
    const bool blk83 = OBS_MODE != CBEV_OBS_RGB && P.blk83 != 0;
    // blocks under the ego square [eg0, eg0 + hero_w) on both axes, as inclusive block ranges
    const int eg0x = P.anchor_x - (P.hero_w >> 1), eg0y = P.anchor_y - (P.hero_w >> 1);
    const int ebx0 = max(eg0x, 0) >> 3, ebxn = (min(eg0x + P.hero_w, S) - 1 >> 3) - ebx0;
    const int eby0 = max(eg0y, 0) >> 3, ebyn = (min(eg0y + P.hero_w, S) - 1 >> 3) - eby0;
    // this lane's share of a single-colour block: output (i, j) of its 3 x 3 for the first nine lanes of the block
    const int local = ly * 2 + (lx & 1), loc_i = (local * 11) >> 5;
    const int loc_out = loc_i * P.obs_w + (local - 3 * loc_i) + 3 * (lx >> 1);
    const unsigned mine = (lane & 2) ? 0xccccccccu : 0x33333333u;  // the 16 lanes of this lane's block
    // window byte of texel (x, y): strip (x >> 7) of tile_h rows of 128 bytes, 16-byte chunk ^= row & 7
    const int strip_step = tile_h * BW - BW;
    auto gather_fast = [&](int p) {
      const int oy = (p >> pw_log) * 8 + ly, ox0 = (p & (pw - 1)) * 16 + lx * 4;
      const int ryp = oy - top;
      // the window origin is folded into the 16.16 start values: (d >> 16) - f == (d - (f << 16)) >> 16
      int dx = rax + isin * (rcy - ryp) + (ox0 - left) * icos - (fx << 16);
      int dy = ray - icos * (rcy - ryp) + (ox0 - left) * isin - (fy << 16);
      uint32_t packed = 0;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int x = dx >> 16, y = dy >> 16;
        packed |= (uint32_t)s_tile[(y * BW + (x >> 7) * strip_step + x) ^ ((y << 4) & 0x70)] << (8 * k);
        dx += icos;
        dy += isin;
      }
      return packed;
    };
    auto gather_generic = [&](int p) {
      const int oy = (p >> pw_log) * 8 + ly, ox0 = (p & (pw - 1)) * 16 + lx * 4;
      const int ryp = oy - top;
      const bool row_in = ryp >= 0 && ryp < ny;
      const int bx = rax + isin * (rcy - ryp);
      const int by = ray - icos * (rcy - ryp);
      uint32_t packed = 0;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int rxp = ox0 + k - left;
        uint32_t v = CBEV_PAL_BLACK;
        if (row_in && rxp >= 0 && rxp < nx) {
          if (mode == 0) {
            int sx, sy;
            if (turns == 0) { sx = rxp; sy = ryp; }
            else if (turns == 1) { sx = crop - 1 - ryp; sy = rxp; }
            else if (turns == 2) { sx = crop - 1 - rxp; sy = crop - 1 - ryp; }
            else { sx = ryp; sy = crop - 1 - rxp; }
            v = s_tile[tile_off(sx - s_desc[RD_FX], sy - fy)];
          } else {
            const int dx = bx + rxp * icos, dy = by + rxp * isin;
            if (dx < 0 || dy < 0 || dx > lim || dy > lim) v = bg;
            else v = s_tile[tile_off((dx >> 16) - s_desc[RD_FX], (dy >> 16) - fy)];
          }
        }
        packed |= v << (8 * k);
      }
      return packed;
    };
    // where the four texels of a lane go: the frame, unless their 8 x 8 block is one colour (shortcut above)
    auto finish = [&](int p, uint32_t packed) {
      const int oy = (p >> pw_log) * 8 + ly, ox0 = (p & (pw - 1)) * 16 + lx * 4;
      bool keep = true;
      if (blk83) {
        const uint32_t c = __shfl_sync(0xffffffffu, packed, lane & 2) & 255u;  // first texel of this lane's block
        const unsigned agree = __ballot_sync(0xffffffffu, packed == c * 0x01010101u);
        const int pxp = p & (pw - 1), by = p >> pw_log, bx = 2 * pxp + (lx >> 1);  // block index = 2 p + (lx >> 1)
        const bool ego = (unsigned)(bx - ebx0) <= (unsigned)ebxn && (unsigned)(by - eby0) <= (unsigned)ebyn;
        const bool uni = (agree & mine) == mine && !ego;
        keep = !uni;
        if (local == 0) s_bflag[2 * p + (lx >> 1)] = uni ? 0 : 1;
        if (uni && local < 9) s_out_sep[3 * by * P.obs_w + 6 * pxp + loc_out] = s_cmu[c];
      }
      if (keep) *(uint32_t*)(s_fov + oy * FP + ox0) = packed;
    };
    if (fast) {
      // four patches per iteration: all sixteen gathers of a lane are issued before the first of them is consumed
      // (npatch / nwarps is 4 at S = 64 and 16 at S = 128 / 256)
#pragma unroll 1
      for (int p = warp; p < npatch; p += 4 * nwarps) {
        uint32_t pk[4];
#pragma unroll
        for (int g = 0; g < 4; ++g) pk[g] = gather_fast(p + g * nwarps);
#pragma unroll
        for (int g = 0; g < 4; ++g) finish(p + g * nwarps, pk[g]);
      }
    } else {
      for (int p = warp; p < npatch; p += nwarps) finish(p, gather_generic(p));
    }
    __syncthreads();
    if (P.fov_mask != nullptr) {  // apply_mask (fov.py:96-99) before the ego is drawn
      const int wq = S >> 2, wq_log = 31 - __clz(wq);
      for (int u = tid; u < S * wq; u += NT) {
        const uint32_t mk = ((const uint32_t*)P.fov_mask)[u];
        uint32_t* px = (uint32_t*)(s_fov + (u >> wq_log) * FP) + (u & (wq - 1));
        *px = (*px & ~mk) | ((CBEV_PAL_BLACK * 0x01010101u) & mk);
      }
      __syncthreads();
    }
    // Hero.draw: hero_w x hero_w black square, rect centred on the anchor (hero.py:17-32), clipped to the surface
    const int hw = P.hero_w;
    if (tid < hw * hw) {
      const int x = P.anchor_x - (hw >> 1) + tid % hw, y = P.anchor_y - (hw >> 1) + tid / hw;
      if (x >= 0 && x < S && y >= 0 && y < S) s_fov[y * FP + x] = CBEV_PAL_BLACK;
    }
  }
  __syncthreads();
  trace_mark(P, env, 3);
  const int cq = S >> 4, cq_log = 31 - __clz(cq);  // 16-byte chunks per frame row
  if (P.fov_out != nullptr) {
    uint4* dst = (uint4*)(P.fov_out + (size_t)env * S * S);
    for (int u = tid; u < S * cq; u += NT) dst[u] = *(const uint4*)(s_fov + (u >> cq_log) * FP + ((u & (cq - 1)) << 4));
  }

  const int F = P.frame_stack;
  const int first = (flags & 1) ? P.head - F + 1 : P.head;

  if (OBS_MODE == CBEV_OBS_RGB) {
    // raw render(): (S, S, 3) uint8; 16 pixels -> 48 bytes = three 16-byte stores per thread
    uint8_t* dst = (uint8_t*)P.ring + (size_t)env * P.ring_slots * P.frame_bytes + (size_t)P.head * P.frame_bytes;
    for (int u = tid; u < S * cq; u += NT) {
      const uint4 p16 = *(const uint4*)(s_fov + (u >> cq_log) * FP + ((u & (cq - 1)) << 4));
      uint32_t o[12];
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        const uint32_t p4 = (&p16.x)[g];
        const uint32_t k0 = s_key[p4 & 255u], k1 = s_key[(p4 >> 8) & 255u], k2 = s_key[(p4 >> 16) & 255u],
                       k3 = s_key[p4 >> 24];
        o[3 * g] = k0 | (k1 << 24);
        o[3 * g + 1] = (k1 >> 8) | (k2 << 16);
        o[3 * g + 2] = (k2 >> 16) | (k3 << 8);
      }
#pragma unroll
      for (int g = 0; g < 3; ++g) st_b4(dst + 48 * (size_t)u + 16 * g, o[4 * g], o[4 * g + 1], o[4 * g + 2], o[4 * g + 3]);
    }
    return;
  }

  // ---- 4. cv2.resize(INTER_AREA) (ResizeObservation, envs/__init__.py:62) + colour equality / gray level ----
  const int OH = P.obs_h, OW = P.obs_w;
  const bool blk83 = P.blk83 != 0;
  uint8_t* const s_out = blk83 ? s_out_sep : smem;  // the tile is dead
  uint8_t* const s_scratch = blk83 ? smem : smem + ((OH * OW + 15) & ~15);  // work lists, in the dead tile
  {
    const int rs_mode = P.rs_mode == CBEV_RS_FAST96 ? CBEV_RS_TABLE : P.rs_mode;
    // area tables: [nx, ny, xoff[OW+1], yoff[OH+1], xsi[nx], ysi[ny], xalpha[nx], yalpha[ny]]
    // bilinear tables: [0, 0, xofs[OW], yofs[OH], xa0[OW], xa1[OW], yb0[OH], yb1[OH]]
    const int nxt = s_tab[0], nyt = s_tab[1];
    const int32_t* xoff = s_tab + 2;
    const int32_t* yoff = xoff + OW + 1;
    const int32_t* xsi = yoff + OH + 1;
    const int32_t* ysi = xsi + nxt;
    const float* xal = (const float*)(ysi + nyt);
    const float* yal = xal + nxt;
    const int32_t* lxo = s_tab + 2;
    const int32_t* lyo = lxo + OW;
    const int32_t* lxa = lyo + OH;       // [2][OW]
    const int32_t* lyb = lxa + 2 * OW;   // [2][OH]
    // (dy, dx) of output o = tid + i * NT without a division per output
    const int qN = NT / OW, rN = NT - qN * OW;
    if (rs_mode == CBEV_RS_TABLE) {
      // Pass A: an output whose whole source footprint is one colour resolves to that colour (sixteen independent
      // loads, no arithmetic); the others are queued.  Pass B works the queue off with the float32 tables, all lanes
      // busy (as the 4x4-block two-pass resize of k_render does for 128 -> 96).
      const int32_t* fxlo = (const int32_t*)(yal + nyt);
      const int32_t* fxhi = fxlo + OW;
      const int32_t* fylo = fxhi + OW;
      const int32_t* fyhi = fylo + OH;
      uint16_t* s_list = (uint16_t*)s_scratch;
      int* s_count = (int*)(s_bar + 1);  // [0] mixed outputs, [1] flagged blocks
      if (tid < 2) s_count[tid] = 0;
      __syncthreads();
      // one output: single-colour footprint -> s_cmu, otherwise onto the list (warp-aggregated; call it converged)
      auto pass_a = [&](bool valid, int o, int dx, int dy) {
        bool uni = true;
        if (valid) {
          uint32_t c0 = 0;
          const int xl = fxlo[dx], xh = fxhi[dx], yl = fylo[dy], yh = fyhi[dy];
          if (xh - xl < 4 && yh - yl < 4) {
            // footprint of <= 4 x 4: per row one 4-byte window starting at column xl (two aligned words, funnel
            // shift), compared with the first pixel's colour under a mask of the footprint's width
            const int sh8 = (xl & 3) * 8, wlo = xl >> 2, whi = xh >> 2;
            const uint32_t msk = 0xffffffffu >> (8 * (3 - (xh - xl)));
            uint32_t diff = 0, c4 = 0;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const uint32_t* row = (const uint32_t*)(s_fov + min(yl + i, yh) * FP);
              const uint32_t win = __funnelshift_r(row[wlo], row[whi], sh8);
              if (i == 0) { c0 = win & 255u; c4 = c0 * 0x01010101u; }
              diff |= (win ^ c4) & msk;
            }
            uni = diff == 0;
          } else {
            c0 = s_fov[yl * FP + xl];
            for (int yy = yl; yy <= yh; ++yy)
              for (int xx = xl; xx <= xh; ++xx) uni = uni && s_fov[yy * FP + xx] == c0;
          }
          if (uni) s_out[o] = s_cmu[c0];
        }
        const unsigned mixed = __ballot_sync(0xffffffffu, valid && !uni);
        if (mixed) {
          int pos = 0;
          if (lane == 0) pos = atomicAdd(s_count, __popc(mixed));
          pos = __shfl_sync(0xffffffffu, pos, 0);
          if (valid && !uni) s_list[pos + __popc(mixed & ((1u << lane) - 1u))] = (uint16_t)o;
        }
      };
      // (without the block shortcut the outputs go in bands of P.list_cap: the work list of a band always fits the dead
      //  tile, whatever the observation size -- one band for everything up to about 150 x 150 at size 128)
      const int total = OH * OW, band = blk83 ? total : min(total, P.list_cap);
      int nmixed_all = 0;
      for (int b0 = 0; b0 < total; b0 += band) {
        const int b1 = min(b0 + band, total);
        if (b0 > 0) {  // pass B of the previous band is done before its list is reused
          __syncthreads();
          if (tid == 0) s_count[0] = 0;
          __syncthreads();
        }
        if (blk83) {
          // the flagged blocks, compacted; then their nine outputs each
          uint16_t* s_blist = s_list + OH * OW;
          const int nblk = (S >> 3) * (S >> 3), nbw = S >> 3, nbw_log = 31 - __clz(nbw);
          for (int k0 = 0; k0 < nblk; k0 += NT) {
            const int b = k0 + tid;
            const bool flagged = b < nblk && s_bflag[b] != 0;
            const unsigned m = __ballot_sync(0xffffffffu, flagged);
            if (m) {
              int pos = 0;
              if (lane == 0) pos = atomicAdd(s_count + 1, __popc(m));
              pos = __shfl_sync(0xffffffffu, pos, 0);
              if (flagged) s_blist[pos + __popc(m & ((1u << lane) - 1u))] = (uint16_t)b;
            }
          }
          __syncthreads();
          const int n9 = s_count[1] * 9;
          for (int i0 = 0; i0 < n9; i0 += NT) {
            const int idx = i0 + tid;
            const bool valid = idx < n9;
            int o = 0, dx = 0, dy = 0;
            if (valid) {
              const int q = idx / 9, sub = idx - 9 * q, blk = s_blist[q];
              const int by = blk >> nbw_log, bx = blk & (nbw - 1), i = (sub * 11) >> 5;
              dy = 3 * by + i;
              dx = 3 * bx + (sub - 3 * i);
              o = dy * OW + dx;
            }
            pass_a(valid, o, dx, dy);
          }
        } else {
          int dy = (b0 + tid) / OW, dx = (b0 + tid) - dy * OW;
          for (int o0 = b0; o0 < b1; o0 += NT) {  // uniform trip count: the queue is filled with warp ballots
            const int o = o0 + tid;
            pass_a(o < b1, o, dx, dy);
            dy += qN;
            dx += rN;
            if (dx >= OW) { dx -= OW; ++dy; }
          }
        }
        __syncthreads();
        const int nmixed = *s_count;
        nmixed_all += nmixed;
        for (int idx = tid; idx < nmixed; idx += NT) {
          const int o = s_list[idx];
          const int oy = o / OW, ox = o - oy * OW;
          // ResizeArea_Invoker: buf = sum_x S * alpha (from 0, in table order); sum = sum_y beta * buf; float32, no FMA
          float sr = 0.f, sg = 0.f, sb = 0.f;
          const int y0 = yoff[oy], y1 = yoff[oy + 1], x0 = xoff[ox], x1 = xoff[ox + 1];
          if (x1 - x0 <= 4 && y1 - y0 <= 4) {
            // footprint of <= 4 x 4 consecutive texels (every shrink ratio below 3, and 8 : 3): the rows come as the
            // 4-byte windows of pass A, the sums are unrolled; a tap beyond the footprint has weight +0.0f, and
            // x + (+0.0f) = x exactly, so the padded sums are OpenCV's sums
            const int xl = xsi[x0], sh8 = (xl & 3) * 8, wlo = xl >> 2, whi = (xl + (x1 - x0) - 1) >> 2;
            float ax[4];
  #pragma unroll
            for (int k = 0; k < 4; ++k) ax[k] = x0 + k < x1 ? xal[x0 + k] : 0.f;
  #pragma unroll
            for (int j = 0; j < 4; ++j) {
              if (y0 + j < y1) {
                const uint32_t* row = (const uint32_t*)(s_fov + ysi[y0 + j] * FP);
                const uint32_t win = __funnelshift_r(row[wlo], row[whi], sh8);
                float br = 0.f, bg = 0.f, bb = 0.f;
  #pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const float4 c = s_palf[(win >> (8 * k)) & 255u];
                  br = __fadd_rn(br, __fmul_rn(c.x, ax[k]));
                  bg = __fadd_rn(bg, __fmul_rn(c.y, ax[k]));
                  bb = __fadd_rn(bb, __fmul_rn(c.z, ax[k]));
                }
                const float beta = yal[y0 + j];
                sr = __fadd_rn(sr, __fmul_rn(beta, br));
                sg = __fadd_rn(sg, __fmul_rn(beta, bg));
                sb = __fadd_rn(sb, __fmul_rn(beta, bb));
              }
            }
          } else
          for (int j = y0; j < y1; ++j) {
            const uint8_t* srow = s_fov + ysi[j] * FP;
            float br = 0.f, bg = 0.f, bb = 0.f;
            for (int k = x0; k < x1; ++k) {
              const uint32_t kk = s_key[srow[xsi[k]]];
              const float a = xal[k];
              br = __fadd_rn(br, __fmul_rn((float)(kk & 255u), a));
              bg = __fadd_rn(bg, __fmul_rn((float)((kk >> 8) & 255u), a));
              bb = __fadd_rn(bb, __fmul_rn((float)(kk >> 16), a));
            }
            const float beta = yal[j];
            sr = __fadd_rn(sr, __fmul_rn(beta, br));
            sg = __fadd_rn(sg, __fmul_rn(beta, bg));
            sb = __fadd_rn(sb, __fmul_rn(beta, bb));
          }
          const int R = min(max(__float2int_rn(sr), 0), 255), G = min(max(__float2int_rn(sg), 0), 255),
                    B = min(max(__float2int_rn(sb), 0), 255);
          s_out[o] = (uint8_t)classify_key<OBS_MODE>((uint32_t)R | ((uint32_t)G << 8) | ((uint32_t)B << 16), s_key, s_cm);
        }
      }  // bands
      if (P.trace != nullptr && tid == 0)  // work-list sizes for tools/render_trace_any.py: flagged blocks, mixed outputs
        P.trace[(size_t)env * 8 + 7] = (unsigned)s_count[1] | ((unsigned long long)(unsigned)nmixed_all << 32);
    } else {
      // copy / exact halving / enlarging: taps of one colour give that colour exactly in every mode ((4c + 2) >> 2 = c;
      // the bilinear kernel: below) and its output byte is tabulated -- pass A; the outputs with mixed taps are queued
      // with warp ballots and pass B computes them with all lanes busy
      uint16_t* s_list = (uint16_t*)s_scratch;
      int* s_count = (int*)(s_bar + 1);
      if (tid == 0) s_count[0] = 0;
      __syncthreads();
      const bool unit_taps = s_tab[0] == 1;  // bilinear: every tap pair sums to 2048 (api.cu checks)
      const int total = OH * OW, band = min(total, P.list_cap);  // bands: see the table resize
      int nmixed_all = 0;
      for (int b0 = 0; b0 < total; b0 += band) {
        const int b1 = min(b0 + band, total);
        if (b0 > 0) {
          __syncthreads();
          if (tid == 0) s_count[0] = 0;
          __syncthreads();
        }
        int dy = (b0 + tid) / OW, dx = (b0 + tid) - dy * OW;
        for (int o0 = b0; o0 < b1; o0 += NT) {  // uniform trip count
          const int o = o0 + tid;
          const bool valid = o < b1;
          int same = -1;
          if (valid) {
            if (rs_mode == CBEV_RS_COPY) {
              same = s_fov[dy * FP + dx];
            } else if (rs_mode == CBEV_RS_HALF) {
              const uint8_t* q0 = s_fov + (2 * dy) * FP + 2 * dx;
              const uint32_t c0 = q0[0], c1 = q0[1], c2 = q0[FP], c3 = q0[FP + 1];
              if (c0 == c1 && c0 == c2 && c0 == c3) same = (int)c0;
            } else {
              // four equal taps c: floor(b0 c / 512) + floor(b1 c / 512) is 4c - 1 or 4c, and (that + 2) >> 2 = c
              const int sx0 = lxo[dx], sx1 = min(sx0 + 1, S - 1), sy0 = lyo[dy], sy1 = min(sy0 + 1, S - 1);
              const uint32_t i00 = s_fov[sy0 * FP + sx0], i01 = s_fov[sy0 * FP + sx1], i10 = s_fov[sy1 * FP + sx0],
                             i11 = s_fov[sy1 * FP + sx1];
              if (unit_taps && i00 == i01 && i00 == i10 && i00 == i11) same = (int)i00;
            }
            if (same >= 0) s_out[o] = s_cmu[same];
          }
          const unsigned mixed = __ballot_sync(0xffffffffu, valid && same < 0);
          if (mixed) {
            int pos = 0;
            if (lane == 0) pos = atomicAdd(s_count, __popc(mixed));
            pos = __shfl_sync(0xffffffffu, pos, 0);
            if (valid && same < 0) s_list[pos + __popc(mixed & ((1u << lane) - 1u))] = (uint16_t)o;
          }
          dy += qN;
          dx += rN;
          if (dx >= OW) { dx -= OW; ++dy; }
        }
        __syncthreads();
        const int nmixed = s_count[0];
        nmixed_all += nmixed;
        for (int idx = tid; idx < nmixed; idx += NT) {
          const int o = s_list[idx];
          const int oy = o / OW, ox = o - oy * OW;
          uint32_t key = 0;
          if (rs_mode == CBEV_RS_HALF) {
            // OpenCV's 2x2 fast path for 8-bit images: (a + b + c + d + 2) >> 2 per channel
            const uint8_t* q0 = s_fov + (2 * oy) * FP + 2 * ox;
            const uint32_t c0 = q0[0], c1 = q0[1], c2 = q0[FP], c3 = q0[FP + 1];
            const uint32_t rg = s_rg[c0] + s_rg[c1] + s_rg[c2] + s_rg[c3] + 0x00020002u;
            const uint32_t b = s_b[c0] + s_b[c1] + s_b[c2] + s_b[c3] + 2u;
            key = ((rg & 0xffffu) >> 2) | ((rg >> 18) << 8) | ((b >> 2) << 16);
          } else {
            // CBEV_RS_LINEAR.  HResizeLinear: int32 rows = S0 * a0 + S1 * a1;
            // VResizeLinear: ((b0 * (r0 >> 4)) >> 16) + ((b1 * (r1 >> 4)) >> 16) + 2 >> 2
            const int sx0 = lxo[ox], sx1 = min(sx0 + 1, S - 1), sy0 = lyo[oy], sy1 = min(sy0 + 1, S - 1);
            const int a0 = lxa[ox], a1 = lxa[OW + ox], b0 = lyb[oy], b1 = lyb[OH + oy];
            const uint32_t k00 = s_key[s_fov[sy0 * FP + sx0]], k01 = s_key[s_fov[sy0 * FP + sx1]],
                           k10 = s_key[s_fov[sy1 * FP + sx0]], k11 = s_key[s_fov[sy1 * FP + sx1]];
  #pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
              const int r0 = (int)((k00 >> (8 * ch)) & 255u) * a0 + (int)((k01 >> (8 * ch)) & 255u) * a1;
              const int r1 = (int)((k10 >> (8 * ch)) & 255u) * a0 + (int)((k11 >> (8 * ch)) & 255u) * a1;
              const int v = (((b0 * (r0 >> 4)) >> 16) + ((b1 * (r1 >> 4)) >> 16) + 2) >> 2;
              key |= (uint32_t)min(max(v, 0), 255) << (8 * ch);
            }
          }
          s_out[o] = (uint8_t)classify_key<OBS_MODE>(key, s_key, s_cm);
        }
      }  // bands
      if (P.trace != nullptr && tid == 0) P.trace[(size_t)env * 8 + 7] = (unsigned long long)(unsigned)nmixed_all << 32;
    }
  }
  __syncthreads();

  // ---- 5. expand + stream out (as k_render) ----
  trace_mark(P, env, 4);
  for (int slot = first; slot <= P.head; ++slot) {
#pragma unroll 1
    for (int rep = 0; rep < 2; ++rep) {
      int sl = slot;
      if (rep == 1) {
        sl = slot - P.mirror;
        if (P.mirror <= 0 || sl < 0) break;
      }
      uint8_t* base = (uint8_t*)P.ring + ((size_t)env * P.ring_slots + sl) * P.frame_bytes;
      if (U8) {
        store_u8_planes<CHANNELS>(base, s_out, OH * OW, tid, NT);
      } else if (OBS_MODE == CBEV_OBS_SEMANTIC) {
        float* fb = (float*)base;
        const int plane = OH * OW;
        for (int q = tid; q < plane / 4; q += NT) {
          const uint32_t m4 = ((const uint32_t*)s_out)[q];
#pragma unroll
          for (int c = 0; c < CHANNELS; ++c)
            st_b4(fb + c * plane + 4 * q, bit_to_f32(m4, c), bit_to_f32(m4, c + 8), bit_to_f32(m4, c + 16),
                  bit_to_f32(m4, c + 24));
        }
      } else {
        for (int q = tid; q < OH * OW / 16; q += NT) st_u4(base + 16 * q, ((const uint4*)s_out)[q]);
      }
    }
  }
  trace_mark(P, env, 5);
}

// ---- temporal fusion of the stacked masks (wrappers/rgb_to_semantic.py:152-193) ---------------------
// One thread per 16-byte vector V of one output plane -- a float4 of a float32 ring, 16 pixels of a uint8 ring;
// planes are gathered from the ring window.  OutT is the output element: the ring's for a copied plane, float for the
// weighted vehicle history of a uint8 ring (whose other planes are then widened to 0.0f / 1.0f).
__device__ __forceinline__ float weighted3(float a, float b, float d) {
  // float32: ((0 + 1.0 a) + 0.5 b) + 0.25 d, then clip to [0, 1]
  return fminf(fmaxf(__fadd_rn(__fadd_rn(a, __fmul_rn(0.5f, b)), __fmul_rn(0.25f, d)), 0.f), 1.f);
}
__device__ __forceinline__ float u8_lane(const uint4& v, int k) { return (float)(((&v.x)[k >> 2] >> (8 * (k & 3))) & 255u); }

template <typename V, typename OutT>
__global__ void __launch_bounds__(256)
k_fuse(const V* __restrict__ ring, OutT* __restrict__ out, int N, int L, int C, int head, int veh, int mode,
       int HWV) {
  constexpr bool RING_U8 = std::is_same<V, uint4>::value;
  const int Cout = mode == CBEV_FUSE_VEHICLE_TEMPORAL ? C - 1 + 3 : C;
  const long long total = (long long)N * Cout * HWV;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int q = (int)(i % HWV);
    const int c = (int)((i / HWV) % Cout);
    const int env = (int)(i / ((long long)HWV * Cout));
    const V* frame = ring + ((size_t)env * L + head) * C * HWV;  // newest frame
    if (c == C - 1 && mode == CBEV_FUSE_VEHICLE_WEIGHTED) {
      const V a = frame[(size_t)veh * HWV + q];
      const V b = (frame - (size_t)C * HWV)[(size_t)veh * HWV + q];
      const V d = (frame - (size_t)2 * C * HWV)[(size_t)veh * HWV + q];
      if constexpr (RING_U8) {
        float* o = (float*)out + 16 * i;
#pragma unroll
        for (int g = 0; g < 4; ++g)
          st_f4(o + 4 * g, weighted3(u8_lane(a, 4 * g), u8_lane(b, 4 * g), u8_lane(d, 4 * g)),
                weighted3(u8_lane(a, 4 * g + 1), u8_lane(b, 4 * g + 1), u8_lane(d, 4 * g + 1)),
                weighted3(u8_lane(a, 4 * g + 2), u8_lane(b, 4 * g + 2), u8_lane(d, 4 * g + 2)),
                weighted3(u8_lane(a, 4 * g + 3), u8_lane(b, 4 * g + 3), u8_lane(d, 4 * g + 3)));
      } else {
        st_f4((float*)out + 4 * i, weighted3(a.x, b.x, d.x), weighted3(a.y, b.y, d.y), weighted3(a.z, b.z, d.z),
              weighted3(a.w, b.w, d.w));
      }
      continue;
    }
    V v;
    if (c < C - 1) {
      const int src = c < veh ? c : c + 1;  // np.delete(current, vehicle_idx, axis=0)
      v = frame[(size_t)src * HWV + q];
    } else {
      const int age = c - (C - 1);          // history[::-1]: t, t-1, t-2
      v = (frame - (size_t)age * C * HWV)[(size_t)veh * HWV + q];
    }
    if constexpr (!RING_U8) {
      st_f4((float*)out + 4 * i, v.x, v.y, v.z, v.w);
    } else if constexpr (sizeof(OutT) == 1) {
      st_u4((uint8_t*)out + 16 * i, v);
    } else {
      float* o = (float*)out + 16 * i;
#pragma unroll
      for (int g = 0; g < 4; ++g) st_f4(o + 4 * g, u8_lane(v, 4 * g), u8_lane(v, 4 * g + 1), u8_lane(v, 4 * g + 2), u8_lane(v, 4 * g + 3));
    }
  }
}

// per-device state: the constant tables and the dynamic shared-memory opt-in belong to a device / context
constexpr int MAX_DEVICES = 64;
bool g_tables_ready[MAX_DEVICES] = {};

void upload_tables() {
  static const uint8_t pal[CBEV_PAL_COUNT][3] = {{150, 150, 150}, {255, 255, 255}, {220, 220, 220}, {0, 7, 175},
                                                 {255, 0, 0},     {0, 255, 0},     {255, 64, 64},    {255, 255, 0},
                                                 {0, 0, 0},       {100, 100, 100}};  // semantics.py:19-28
  uint32_t rg[CBEV_PAL_COUNT], b[CBEV_PAL_COUNT], key[CBEV_PAL_COUNT];
  for (int i = 0; i < CBEV_PAL_COUNT; ++i) {
    rg[i] = pal[i][0] | ((uint32_t)pal[i][1] << 16);
    b[i] = pal[i][2];
    key[i] = pal[i][0] | ((uint32_t)pal[i][1] << 8) | ((uint32_t)pal[i][2] << 16);
  }
  // channel membership per mask mode (wrappers/rgb_to_semantic.py:6-42); "drivable" = white or green
  uint8_t cm[6][CBEV_PAL_COUNT + 1] = {};
  const int ND = CBEV_PAL_NON_DRIVABLE, DR = CBEV_PAL_DRIVABLE, SW = CBEV_PAL_SIDEWALK, VE = CBEV_PAL_VEHICLE,
            PE = CBEV_PAL_PEDESTRIAN, RO = CBEV_PAL_ROUTE, TL = CBEV_PAL_TL_RED;
  cm[CBEV_MASK_BINARY][DR] = 1; cm[CBEV_MASK_BINARY][RO] = 1;
  cm[CBEV_MASK_2][DR] = 1; cm[CBEV_MASK_2][RO] = 1 | 2;
  cm[CBEV_MASK_4][DR] = 1; cm[CBEV_MASK_4][VE] = 2; cm[CBEV_MASK_4][PE] = 4; cm[CBEV_MASK_4][RO] = 1 | 8;
  cm[CBEV_MASK_5][DR] = 1; cm[CBEV_MASK_5][SW] = 2; cm[CBEV_MASK_5][VE] = 4; cm[CBEV_MASK_5][PE] = 8;
  cm[CBEV_MASK_5][RO] = 1 | 16;
  for (int m = CBEV_MASK_6; m <= CBEV_MASK_7; ++m) {
    cm[m][ND] = 1; cm[m][DR] = 2; cm[m][SW] = 4; cm[m][VE] = 8; cm[m][PE] = 16; cm[m][RO] = 2 | 32;
  }
  cm[CBEV_MASK_7][TL] = 64;
  cudaMemcpyToSymbol(c_pal_rg, rg, sizeof(rg));
  cudaMemcpyToSymbol(c_pal_b, b, sizeof(b));
  cudaMemcpyToSymbol(c_pal_key, key, sizeof(key));
  cudaMemcpyToSymbol(c_chan_mask, cm, sizeof(cm));
}

template <int MODE, int CH, bool U8 = false>
int launch(cbev_engine* e, const RenderParams& P, size_t smem, size_t smem_any, bool any, cudaStream_t s) {
  static bool attr_done[MAX_DEVICES][2] = {};
  const int dev = e->device >= 0 && e->device < MAX_DEVICES ? e->device : 0;
  if (any) {
    auto kern = k_render_any<MODE, CH, U8>;
    if (!attr_done[dev][1]) {
      if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess) {
        cbev_set_error("k_render_any: cannot opt in to 227 KB of dynamic shared memory: %s",
                       cudaGetErrorString(cudaGetLastError()));
        return 1;
      }
      attr_done[dev][1] = true;
    }
    kern<<<P.N, P.fov > 128 ? 1024 : 256, smem_any, s>>>(P, *reinterpret_cast<const CUtensorMap*>(e->tmap_any),
                                                        e->cfg.mask_mode);
    return 0;
  }
  auto kern = k_render<MODE, CH, U8>;
  if (!attr_done[dev][0]) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024) != cudaSuccess) {
      cbev_set_error("k_render: cannot opt in to 100 KB of dynamic shared memory: %s",
                     cudaGetErrorString(cudaGetLastError()));
      return 1;
    }
    attr_done[dev][0] = true;
  }
  kern<<<P.N, RT, smem, s>>>(P, *reinterpret_cast<const CUtensorMap*>(e->tmap), e->cfg.mask_mode);
  return 0;
}

// the semantic masks: float32 planes, or 0 / 1 byte planes (U8 = CBEV_OBS_SEMANTIC_U8)
template <bool U8>
int launch_semantic(cbev_engine* e, const RenderParams& P, size_t smem, size_t smem_any, bool any, cudaStream_t s) {
  switch (e->channels) {
    case 1: return launch<CBEV_OBS_SEMANTIC, 1, U8>(e, P, smem, smem_any, any, s);
    case 2: return launch<CBEV_OBS_SEMANTIC, 2, U8>(e, P, smem, smem_any, any, s);
    case 4: return launch<CBEV_OBS_SEMANTIC, 4, U8>(e, P, smem, smem_any, any, s);
    case 5: return launch<CBEV_OBS_SEMANTIC, 5, U8>(e, P, smem, smem_any, any, s);
    case 6: return launch<CBEV_OBS_SEMANTIC, 6, U8>(e, P, smem, smem_any, any, s);
    case 7: return launch<CBEV_OBS_SEMANTIC, 7, U8>(e, P, smem, smem_any, any, s);
    default: cbev_set_error("no raster kernel for %d mask channels", e->channels); return 1;
  }
}

// What the live step and the lookahead leaf windows share: the constant tables, everything of RenderParams but the
// grid (N), the descriptor / draw-list / ring pointers, the ring geometry and the step-only outputs (CTA order and its
// counters, kept palette frame, trace), the shared-memory sizes and the choice of kernel.  Then the launch.
int render_launch(cbev_engine* e, RenderParams& P, cudaStream_t s) {
  {
    const int dev = e->device >= 0 && e->device < MAX_DEVICES ? e->device : 0;
    if (!g_tables_ready[dev]) {
      upload_tables();
      g_tables_ready[dev] = true;
    }
  }
  P.fov = e->cfg.fov_size;
  P.crop = e->crop;
  P.anchor_x = e->anchor_x;
  P.anchor_y = e->anchor_y;
  P.frame_stack = e->cfg.frame_stack;
  P.frame_bytes = e->frame_bytes;
  P.max_rects = e->max_rects;
  P.fov_mask = e->fov_mask;
  const int S = P.fov;
  const size_t tile = (size_t)CBEV_TILE_W * CBEV_TILE_H;  // >= 96*96 output bytes + 2*32*32 (mixed-block worklist)
  P.generic_rotate = (e->debug_flags & CBEV_DBG_GENERIC_ROTATE) != 0;
  P.obs_h = e->cfg.obs_h;
  P.obs_w = e->cfg.obs_w;
  P.rs_mode = e->rs_mode;
  P.rs_words = e->rs_words;
  P.rs_tab = e->rs_tab;
  P.hero_w = 32 / (1024 / S);
  P.nbx = e->any_nbx;
  P.nby = e->any_nby;
  P.box_h = e->any_box_h;
  // k_render: size 128 with the (96, 96) observation or the raw frame; everything else (and debug flag 256) k_render_any
  const bool any = S != 128 || (e->cfg.obs_mode != CBEV_OBS_RGB && e->rs_mode != CBEV_RS_FAST96) ||
                   (e->debug_flags & CBEV_DBG_RENDER_ANY);
  const size_t rects_bytes = (size_t)((e->max_rects * CBEV_RECT_WORDS + 3) & ~3) * 4;
  const size_t smem = tile + (size_t)S * S + 3 * 16 * 4 + CBEV_DESC_WORDS * 4 + 16 + 16 + 16 + rects_bytes;
  size_t region = (size_t)CBEV_ANY_BOX_W * P.nbx * P.box_h * P.nby;
  // output bytes + the work list of mixed outputs (uint16 each) of the two-pass resize.  The list need not hold every
  // output: the resize runs in bands of list_cap outputs (>= 4096, or all of them when they are fewer)
  const size_t ohw = (size_t)e->cfg.obs_h * e->cfg.obs_w, ohw16 = (ohw + 15) & ~(size_t)15;
  const size_t out_bytes = ohw16 + 2 * (ohw < 4096 ? ohw : 4096) + 16;
  // 8:3 block shortcut of k_render_any (256 -> 96, 128 -> 48, 64 -> 24): needs the whole-frame passes off (corner mask,
  // debug copy of the frame); debug flag 512 switches it off (A/B probe)
  const size_t nblk = (size_t)(S / 8) * (S / 8);
  P.blk83 = e->cfg.obs_mode != CBEV_OBS_RGB && e->rs_mode == CBEV_RS_TABLE && 3 * S == 8 * e->cfg.obs_w &&
            3 * S == 8 * e->cfg.obs_h && e->fov_mask == nullptr && !e->keep_fov &&
            !(e->debug_flags & CBEV_DBG_NO_BLOCK83);
  if (P.blk83 && 2 * ohw + 2 * nblk + 16 > region) P.blk83 = 0;  // (its lists: nine outputs per flagged block + the blocks)
  if (e->cfg.obs_mode != CBEV_OBS_RGB && out_bytes > region) region = out_bytes;
  P.region_bytes = (int32_t)region;  // a multiple of 1024 (strips) or of 16 (output bytes)
  {
    const size_t room = region > ohw16 + 16 ? (region - ohw16 - 16) / 2 : 0;
    P.list_cap = (int32_t)(room < ohw ? room : ohw);
  }
  size_t sep_bytes = P.blk83 ? ((nblk + 15) & ~(size_t)15) + (((size_t)e->cfg.obs_h * e->cfg.obs_w + 15) & ~(size_t)15) : 0;
  size_t smem_any = region + (size_t)S * (S + 16) + 3 * 16 * 4 + CBEV_DESC_WORDS * 4 + 16 + 16 + 16 + 16 * 16 + rects_bytes +
                    (size_t)e->rs_words * 4;
  if (smem_any + sep_bytes > 227 * 1024) {  // a long draw list at size 256: no room for the shortcut's own output bytes
    P.blk83 = 0;
    sep_bytes = 0;
  }
  smem_any += sep_bytes;
  if (any && smem_any > 227 * 1024) {
    cbev_set_error("k_render_any needs %zu bytes of shared memory (max_rects %d): over the 227 KB of one CTA", smem_any,
                   e->max_rects);
    return 1;
  }
  int rc = 1;
  if (e->cfg.obs_mode == CBEV_OBS_RGB) rc = launch<CBEV_OBS_RGB, 1>(e, P, smem, smem_any, any, s);
  else if (e->cfg.obs_mode == CBEV_OBS_GRAY) rc = launch<CBEV_OBS_GRAY, 1>(e, P, smem, smem_any, any, s);
  else if (e->cfg.obs_mode == CBEV_OBS_SEMANTIC_U8) rc = launch_semantic<true>(e, P, smem, smem_any, any, s);
  else rc = launch_semantic<false>(e, P, smem, smem_any, any, s);
  if (rc == 0) e->launches += 1;
  return rc;
}

}  // namespace

int cbev_launch_render(cbev_engine* e, int32_t head, int32_t mirror, cudaStream_t s) {
  RenderParams P;
  P.N = e->N;
  P.ring_slots = e->cfg.ring_slots;
  P.head = head;
  P.mirror = mirror;
  P.desc = e->desc;
  P.rects = e->rects;
  P.order = (e->debug_flags & CBEV_DBG_IDENTITY_RENDER_ORDER) ? nullptr : e->order;
  P.order_cnt = e->order_cnt;
  P.fov_out = e->keep_fov ? e->fov : nullptr;
  P.ring = e->ring;
  P.trace = (e->debug_flags & CBEV_DBG_TRACE) ? e->trace : nullptr;
  return render_launch(e, P, s);
}

// The leaf windows of cbev_lookahead_obs: render position i (= b * F + f) is a "virtual env" whose one-slot ring row is
// frame f of window b.  No CTA order, no counters to zero, no kept frame, no trace: the live step's state is not read
// or written.  Positions with a skip header (RD_FLAGS bit 1) exit at once.
int cbev_launch_render_branches(cbev_engine* e, int32_t n, void* windows, cudaStream_t s) {
  RenderParams P;
  P.N = n;
  P.ring_slots = 1;
  P.head = 0;
  P.mirror = 0;
  P.desc = e->br_desc;
  P.rects = e->br_rects;
  P.order = nullptr;
  P.order_cnt = nullptr;
  P.fov_out = nullptr;
  P.ring = windows;
  P.trace = nullptr;
  return render_launch(e, P, s);
}

int cbev_launch_fuse(cbev_engine* e, int32_t mode, const void* ring, int32_t n, int32_t L, int32_t head, void* out,
                     cudaStream_t s) {
  // vehicle channel index per mask mode (wrappers/rgb_to_semantic.py:6-62); binary / 2-class have none
  static const int veh_of[6] = {-1, -1, 1, 2, 3, 3};
  const int veh = veh_of[e->cfg.mask_mode];
  if (veh < 0) return 1;
  const int C = e->channels;
  const int Cout = mode == CBEV_FUSE_VEHICLE_TEMPORAL ? C - 1 + 3 : C;
  const bool u8 = e->cfg.obs_mode == CBEV_OBS_SEMANTIC_U8;
  const int HWV = e->cfg.obs_h * e->cfg.obs_w / (u8 ? 16 : 4);  // 16-byte vectors per plane
  long long total = (long long)n * Cout * HWV;
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 32) blocks = 148 * 32;
  if (!u8)
    k_fuse<<<blocks, 256, 0, s>>>((const float4*)ring, (float*)out, n, L, C, head, veh, mode, HWV);
  else if (mode == CBEV_FUSE_VEHICLE_TEMPORAL)
    k_fuse<<<blocks, 256, 0, s>>>((const uint4*)ring, (uint8_t*)out, n, L, C, head, veh, mode, HWV);
  else
    k_fuse<<<blocks, 256, 0, s>>>((const uint4*)ring, (float*)out, n, L, C, head, veh, mode, HWV);
  e->launches += 1;
  return 0;
}

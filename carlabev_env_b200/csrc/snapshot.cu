// snapshot.cu -- k_snapshot / k_restore: whole-env state <-> caller-owned snapshot rows (cbev_snapshot / cbev_restore).
//
// Grid = (chunk, row).  Chunk 0 of a row moves the small per-env state (header + 16 SoA sections, a few hundred
// bytes); chunks 1.. move the F window frames, which are almost all of the bytes (884,736 per env for 6 x 96 x 96
// float32 masks with F = 4), as uint4s: every frame is a 16-byte multiple at a 16-byte aligned ring slot, and every
// row section starts 16-byte aligned.  The state side of the SoA sections ([N][A] per field) is element aligned
// only, so those are copied element by element -- they are < 0.5 % of a row.
#include "engine.h"

namespace {

constexpr int SNAP_THREADS = 256;
constexpr int SNAP_VEC = 4;                               // uint4 per thread and chunk, loaded before any is stored
constexpr int SNAP_CHUNK = SNAP_THREADS * SNAP_VEC;       // uint4 per chunk (16 KB)

struct SnapArgs {
  SnapLayout L;                                  // row side (restore: at the rows' retreat slots)
  uint8_t* base[CBEV_STATE_SECTIONS];             // engine side: SoA arrays
  int32_t state_count[CBEV_STATE_SECTIONS];       // engine side: elements per env (stride)
  int32_t* scene;
  int32_t* episode;
  uint8_t* done;
  uint8_t* ring;
  uint8_t* rows_mem;                             // dst (snapshot) / src (restore)
  const int32_t* env_ids;                        // [n] or null = identity
  const int32_t* rows;                           // [n] or null = identity (restore only)
  int64_t frame_bytes, frame16;
  int32_t N, n, n_rows, F, ring_slots, head, mirror, chunks_per_frame;
};

template <bool RESTORE>
__device__ __forceinline__ void copy_state(const SnapArgs& a, int env, uint8_t* row) {
  const int tid = threadIdx.x;
  if (tid == 0) {
    if (RESTORE) {
      const int4 h = *(const int4*)row;
      a.scene[env] = h.x;
      a.episode[env] = h.y;
      a.done[env] = (uint8_t)h.z;
    } else {
      *(int4*)row = make_int4(a.scene[env], a.episode[env], (int)a.done[env], 0);
    }
  }
#pragma unroll 1
  for (int s = 0; s < CBEV_STATE_SECTIONS; ++s) {
    const int es = a.L.esize[s], nr = a.L.count[s], ns = a.state_count[s];
    uint8_t* rp = row + a.L.off[s];
    uint8_t* sp = a.base[s] + (size_t)env * ns * es;
    if (RESTORE) {
      // a row taken with fewer retreat slots (the pool grew since): the slots it lacks are zeroed
      for (int i = tid; i < ns; i += SNAP_THREADS) {
        if (i < nr) cbev_copy_elem(sp + (size_t)i * es, rp + (size_t)i * es, es);
        else cbev_zero_elem(sp + (size_t)i * es, es);
      }
    } else {
      for (int i = tid; i < nr; i += SNAP_THREADS) cbev_copy_elem(rp + (size_t)i * es, sp + (size_t)i * es, es);
      const int bytes = nr * es, padded = (bytes + 15) & ~15;
      for (int b = bytes + tid; b < padded; b += SNAP_THREADS) rp[b] = 0;
    }
  }
}

// restore: window frame k goes to slot w_k = head - F + 1 + k and, when F > 1 and w_k >= L - F + 1, also to the mirror
// slot w_k - (L - F + 1) -- the slot rule of the raster kernel's reset frames and of cbev_step's mirror write.
// LEAF (leaf rows of cbev_lookahead_ex): the "envs" are the branch rows and the "ring" the [B][F] leaf windows (one
// window of F slots per branch, head F - 1); a branch without a valid root (scene -1) is skipped.
template <bool RESTORE, bool LEAF = false>
__device__ __forceinline__ void snapshot_rows(const SnapArgs& a) {
  const int chunk = blockIdx.x;
  const int k = chunk > 0 ? (chunk - 1) / a.chunks_per_frame : 0;
  const int64_t q0 = chunk > 0 ? (int64_t)((chunk - 1) % a.chunks_per_frame) * SNAP_CHUNK : 0;
  const int slot = a.head - a.F + 1 + k;
  const int mslot = (a.F > 1 && slot >= a.mirror) ? slot - a.mirror : -1;
  for (int i = blockIdx.y; i < a.n; i += gridDim.y) {
    const int env = a.env_ids ? a.env_ids[i] : i;
    const int r = (RESTORE && a.rows) ? a.rows[i] : i;
    if (env < 0 || env >= a.N || r < 0 || r >= a.n_rows) continue;  // device indices are trusted; never out of bounds
    if (LEAF && a.scene[env] < 0) continue;
    uint8_t* row = a.rows_mem + (size_t)r * a.L.row_bytes;
    if (chunk == 0) {
      copy_state<RESTORE>(a, env, row);
      continue;
    }
    uint4* rf = (uint4*)(row + a.L.frames_off + (size_t)k * a.frame_bytes);
    uint4* sf = (uint4*)(a.ring + ((size_t)env * a.ring_slots + slot) * a.frame_bytes);
    uint4 v[SNAP_VEC];
    if (RESTORE) {
      uint4* mf = mslot >= 0 ? (uint4*)(a.ring + ((size_t)env * a.ring_slots + mslot) * a.frame_bytes) : nullptr;
#pragma unroll
      for (int j = 0; j < SNAP_VEC; ++j) {
        const int64_t q = q0 + j * SNAP_THREADS + threadIdx.x;
        if (q < a.frame16) v[j] = rf[q];  // repeated rows (cloning) hit in L2
      }
#pragma unroll
      for (int j = 0; j < SNAP_VEC; ++j) {
        const int64_t q = q0 + j * SNAP_THREADS + threadIdx.x;
        if (q < a.frame16) {
          sf[q] = v[j];
          if (mf) mf[q] = v[j];
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < SNAP_VEC; ++j) {
        const int64_t q = q0 + j * SNAP_THREADS + threadIdx.x;
        if (q < a.frame16) v[j] = sf[q];
      }
#pragma unroll
      for (int j = 0; j < SNAP_VEC; ++j) {
        const int64_t q = q0 + j * SNAP_THREADS + threadIdx.x;
        if (q < a.frame16) __stcs(rf + q, v[j]);  // rows are not read back soon: stream them past L2
      }
    }
  }
}

SnapArgs make_args(cbev_engine* e, EnvState& st, const SnapLayout& L, int32_t n, const int32_t* env_ids) {
  SnapArgs a;
  a.L = L;
  const int32_t A = e->cfg.max_actors > 0 ? e->cfg.max_actors : 1;
  const StateSections S = cbev_state_sections(st, A, e->pool.max_retreat);
  for (int s = 0; s < CBEV_STATE_SECTIONS; ++s) {
    a.base[s] = (uint8_t*)*S.field[s];
    a.state_count[s] = S.count[s];
  }
  a.scene = st.scene;
  a.episode = st.episode;
  a.done = st.done;
  a.ring = (uint8_t*)e->ring;
  a.rows_mem = nullptr;
  a.env_ids = env_ids;
  a.rows = nullptr;
  a.frame_bytes = e->frame_bytes;
  a.frame16 = e->frame_bytes / 16;
  a.N = e->N;
  a.n = n;
  a.n_rows = n;
  a.F = e->cfg.frame_stack;
  a.ring_slots = e->cfg.ring_slots;
  a.head = e->head;
  a.mirror = a.F > 1 ? a.ring_slots - a.F + 1 : 0;
  a.chunks_per_frame = (int32_t)((a.frame16 + SNAP_CHUNK - 1) / SNAP_CHUNK);
  return a;
}

__global__ void __launch_bounds__(SNAP_THREADS) k_snapshot(const SnapArgs a) { snapshot_rows<false>(a); }
__global__ void __launch_bounds__(SNAP_THREADS) k_restore(const SnapArgs a) { snapshot_rows<true>(a); }
__global__ void __launch_bounds__(SNAP_THREADS) k_leaf_rows(const SnapArgs a) { snapshot_rows<false, true>(a); }

// Leaf windows of cbev_lookahead_obs, the part that comes from the root: window position f < F - min(steps[b], F) of
// branch b is frame f + steps[b] of its root's current window (ring slot head - F + 1 + f + steps[b]), copied as it
// is, reset and mirror-zone frames included; a root outside [0, N) (steps = 0) gets a zero window.  The positions
// from f = F - min(steps, F) on belong to the raster launch and are not touched.  Grid = (window position, branch),
// each CTA moving its whole frame in 16 KB chunks of 16-byte vectors as k_snapshot does: most positions usually
// belong to the raster launch, and one CTA per chunk made those empty CTAs cost more than the copies (B200, c2).
struct LeafArgs {
  const uint8_t* ring;
  uint8_t* windows;        // [B][F][frame_bytes]
  const int32_t* roots;    // [B] or null = identity
  const int32_t* steps;    // [B]
  int64_t frame_bytes, frame16;
  int32_t N, B, F, ring_slots, head;
  // ROWS (roots from snapshot rows): frame f + steps of root row r is at rows + r * row_bytes + frames_off
  const uint8_t* rows;
  int64_t row_bytes, frames_off;
  int32_t n_rows, n_scenes;
};

template <bool ROWS>
__device__ __forceinline__ void leaf_window(const LeafArgs& a) {
  const int k = blockIdx.x;  // window position
  for (int b = blockIdx.y; b < a.B; b += gridDim.y) {
    const int st = a.steps[b];
    if (k >= a.F - (st < a.F ? st : a.F)) continue;
    const int root = a.roots ? a.roots[b] : b;
    bool valid;
    const uint8_t* row = nullptr;
    if constexpr (ROWS) {
      // the bounds of k_lookahead_ex's row roots: a row outside [0, n_rows) or with a scene outside the pool is no root
      valid = root >= 0 && root < a.n_rows;
      row = a.rows + (size_t)(valid ? root : 0) * a.row_bytes;
      if (valid) {
        const int scene = *(const int32_t*)row;
        valid = scene >= 0 && scene < a.n_scenes;
      }
    } else {
      valid = root >= 0 && root < a.N;
    }
    uint4* wf = (uint4*)(a.windows + ((size_t)b * a.F + k) * a.frame_bytes);
    const uint4* rf =
        ROWS ? (const uint4*)(row + a.frames_off + (size_t)(k + st) * a.frame_bytes)
             : (const uint4*)(a.ring + ((size_t)(valid ? root : 0) * a.ring_slots + a.head - a.F + 1 + k + st) *
                                           a.frame_bytes);
    for (int64_t q0 = 0; q0 < a.frame16; q0 += SNAP_CHUNK) {
      uint4 v[SNAP_VEC];
#pragma unroll
      for (int j = 0; j < SNAP_VEC; ++j) {
        const int64_t q = q0 + j * SNAP_THREADS + threadIdx.x;
        v[j] = make_uint4(0, 0, 0, 0);
        if (valid && q < a.frame16) v[j] = rf[q];  // repeated roots hit in L2
      }
#pragma unroll
      for (int j = 0; j < SNAP_VEC; ++j) {
        const int64_t q = q0 + j * SNAP_THREADS + threadIdx.x;
        if (q < a.frame16) wf[q] = v[j];
      }
    }
  }
}

__global__ void __launch_bounds__(SNAP_THREADS) k_leaf_window(const LeafArgs a) { leaf_window<false>(a); }
// root windows from snapshot rows: frame f + steps[b] of the row's frame section
__global__ void __launch_bounds__(SNAP_THREADS) k_leaf_window_rows(const LeafArgs a) { leaf_window<true>(a); }

dim3 grid_of(const SnapArgs& a) {
  return dim3((unsigned)(1 + a.F * a.chunks_per_frame), (unsigned)(a.n < 65535 ? a.n : 65535));
}

int64_t align16(int64_t b) { return (b + 15) & ~(int64_t)15; }

}  // namespace

// The last two sections (retreat routes, retreat_n) are sized by R: a row's layout is a function of (A, R, F, frame_bytes).
SnapLayout cbev_snap_layout(const cbev_engine* e, int32_t R) {
  SnapLayout L;
  const int32_t A = e->cfg.max_actors > 0 ? e->cfg.max_actors : 1;
  EnvState none;
  const StateSections S = cbev_state_sections(none, A, R);
  int64_t off = 16;  // header
  for (int s = 0; s < CBEV_STATE_SECTIONS; ++s) {
    L.off[s] = off;
    L.esize[s] = S.esize[s];
    L.count[s] = S.count[s];
    off += align16((int64_t)S.esize[s] * S.count[s]);
  }
  L.frames_off = off;
  L.row_bytes = L.frames_off + (int64_t)e->cfg.frame_stack * e->frame_bytes;
  return L;
}

void cbev_launch_snapshot(cbev_engine* e, const int32_t* env_ids, int32_t n, void* dst, cudaStream_t s) {
  SnapArgs a = make_args(e, e->st, cbev_snap_layout(e, e->pool.max_retreat), n, env_ids);
  a.rows_mem = (uint8_t*)dst;
  k_snapshot<<<grid_of(a), SNAP_THREADS, 0, s>>>(a);
  e->launches += 1;
}

void cbev_launch_restore(cbev_engine* e, const SnapLayout& L, const void* src, int32_t n_rows, const int32_t* rows,
                         const int32_t* env_ids, int32_t n, cudaStream_t s) {
  SnapArgs a = make_args(e, e->st, L, n, env_ids);
  a.rows_mem = (uint8_t*)const_cast<void*>(src);
  a.rows = rows;
  a.n_rows = n_rows;
  k_restore<<<grid_of(a), SNAP_THREADS, 0, s>>>(a);
  e->launches += 1;
}

void cbev_launch_leaf_window(cbev_engine* e, const int32_t* roots, int32_t n_branches, const int32_t* steps,
                             void* windows, const RowSource* src, cudaStream_t s) {
  LeafArgs a;
  a.ring = (const uint8_t*)e->ring;
  a.windows = (uint8_t*)windows;
  a.roots = roots;
  a.steps = steps;
  a.frame_bytes = e->frame_bytes;
  a.frame16 = e->frame_bytes / 16;
  a.N = e->N;
  a.B = n_branches;
  a.F = e->cfg.frame_stack;
  a.ring_slots = e->cfg.ring_slots;
  a.head = e->head;
  a.rows = src ? (const uint8_t*)src->rows : nullptr;
  a.row_bytes = src ? src->L.row_bytes : 0;
  a.frames_off = src ? src->L.frames_off : 0;
  a.n_rows = src ? src->n_rows : 0;
  a.n_scenes = e->pool.n_scenes;
  const dim3 grid((unsigned)a.F, (unsigned)(n_branches < 65535 ? n_branches : 65535));
  if (src) k_leaf_window_rows<<<grid, SNAP_THREADS, 0, s>>>(a);
  else k_leaf_window<<<grid, SNAP_THREADS, 0, s>>>(a);
  e->launches += 1;
}

void cbev_launch_leaf_rows(cbev_engine* e, int32_t n_branches, const void* windows, void* dst, cudaStream_t s) {
  SnapArgs a = make_args(e, e->branch, cbev_snap_layout(e, e->pool.max_retreat), n_branches, nullptr);
  a.ring = (uint8_t*)const_cast<void*>(windows);
  a.ring_slots = a.F;
  a.head = a.F - 1;
  a.N = n_branches;
  a.rows_mem = (uint8_t*)dst;
  k_leaf_rows<<<grid_of(a), SNAP_THREADS, 0, s>>>(a);
  e->launches += 1;
}

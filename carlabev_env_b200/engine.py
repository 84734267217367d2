"""ctypes binding of libcbev.so (include/cbev.h) + a thin torch-tensor front end.

PyTorch is plumbing here: it owns device buffers and streams; every computation of the step
happens inside the hand-written CUDA kernels behind the C ABI.  There is NO CPU fallback: if the
library is missing or no CUDA device is present, constructing an Engine raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build
from .config import CARL_DEFAULTS, SHAPING_DEFAULTS

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libcbev.so")

# enums of include/cbev.h
OBS_SEMANTIC, OBS_GRAY, OBS_RGB, OBS_SEMANTIC_U8 = 0, 1, 2, 3
MASK_DTYPES = ("float32", "uint8")
MASK_MODES = {"binary": 0, "2-class": 1, "4-class": 2, "5-class": 3, "6-class": 4, "7-class": 5}
MASK_CHANNELS = {"binary": 1, "2-class": 2, "4-class": 4, "5-class": 5, "6-class": 6, "7-class": 7}
FUSE_MODES = {"vehicle_temporal": 1, "vehicle_weighted": 2}  # CBEV_FUSE_*
ACTION_DISCRETE, ACTION_CONTINUOUS = 0, 1
REWARD_CARL, REWARD_SHAPING = 0, 1
AUTORESET_DISABLED, AUTORESET_NEXT_STEP = 0, 1
CAUSE_NAMES = (None, "ckpt", "collision", "success", "out_of_bounds", "off_road", "max_actions", "unknown")
HERO_FIELDS = ("x", "y", "yaw", "v", "x_1", "y_1", "yaw_1", "v_1", "dist2wp", "set_point_x", "set_point_y",
               "set_point_yaw", "cmd_gas", "cmd_steer", "cmd_brake", "applied_delta", "speed_mps", "accel_long",
               "accel_lat", "jerk_long", "jerk_lat", "yaw_rate", "yaw_acc", "acc", "target_idx", "hit", "hit_id",
               "tile_class", "n_nearby", "dist2goal", "t", "scene")
EPISODE_FIELDS = ("return", "length", "cause", "mean_speed", "mean_abs_accel_long", "mean_abs_accel_lat",
                  "mean_abs_jerk_long", "mean_abs_jerk_lat", "mean_abs_yaw_rate", "mean_abs_yaw_acc",
                  "comfort_violation_rate", "harsh_brake_rate", "scene", "num_vehicles", "len_ego_route", "episode")
STATS_FIELDS = 4 + 8 + 6 + 3
SG_MAX = 12
EXPORTS = ("cbev_version", "cbev_last_error", "cbev_create", "cbev_destroy", "cbev_upload_map",
           "cbev_upload_scene_pool", "cbev_frame_bytes", "cbev_bind_obs_ring", "cbev_reset", "cbev_step",
           "cbev_step_host", "cbev_obs_head", "cbev_get_state", "cbev_set_ego_state", "cbev_copy_fov",
           "cbev_read_stats", "cbev_launch_count", "cbev_profile_enable", "cbev_profile_read", "cbev_abi_sizes",
           "cbev_keep_fov", "cbev_upload_fov_mask", "cbev_fuse", "cbev_set_debug_flags",
           "cbev_debug_read_trace", "cbev_step_host_ex", "cbev_wait_host_outputs", "cbev_set_state",
           "cbev_profile_read_ex", "cbev_step_ex", "cbev_invalidate", "cbev_generate_scenes", "cbev_pool_counts",
           "cbev_read_scene_pool", "cbev_snapshot_row_bytes", "cbev_snapshot", "cbev_restore", "cbev_lookahead",
           "cbev_lookahead_obs", "cbev_fuse_windows", "cbev_lookahead_ex", "cbev_set_action_repeat")
MAX_ACTION_REPEAT = 64  # CBEV_MAX_ACTION_REPEAT


class CbevConfig(C.Structure):
    _fields_ = [
        ("num_envs", C.c_int32), ("fov_size", C.c_int32),
        ("anchor_x_frac", C.c_double), ("anchor_y_frac", C.c_double),
        ("obs_h", C.c_int32), ("obs_w", C.c_int32), ("obs_mode", C.c_int32), ("mask_mode", C.c_int32),
        ("frame_stack", C.c_int32), ("ring_slots", C.c_int32), ("action_mode", C.c_int32), ("n_discrete", C.c_int32),
        ("discrete_table", C.c_float * 48),
        ("reward_mode", C.c_int32), ("autoreset", C.c_int32), ("max_actors", C.c_int32), ("trajectory_steps", C.c_int32),
        ("lane_center_exponent", C.c_double), ("lane_center_floor", C.c_double), ("off_lane_penalty", C.c_double),
        ("speed_penalty_scale", C.c_double), ("speed_penalty_floor", C.c_double), ("ttc_threshold", C.c_double),
        ("ttc_penalty_floor", C.c_double),
        ("max_actions", C.c_int32), ("offroad_terminate_after", C.c_int32),
        ("sidewalk_step_penalty", C.c_double), ("sidewalk_penalty_scale", C.c_double),
        ("k_lat_quadratic", C.c_double), ("k_progress", C.c_double), ("k_flow", C.c_double),
        ("k_align_bonus", C.c_double), ("k_reverse", C.c_double), ("k_ttc", C.c_double), ("alive_bias", C.c_double),
        ("k_smooth", C.c_double), ("k_steer_smooth", C.c_double), ("k_steer_jerk", C.c_double),
        ("k_route_dev", C.c_double), ("route_dev_start", C.c_double),
        ("max_speed_for_flow", C.c_double), ("lat_clip", C.c_double), ("yaw_small", C.c_double),
        ("lat_small", C.c_double),
        ("seed", C.c_uint64),
    ]


_P = C.c_void_p


class CbevPoolDesc(C.Structure):
    _fields_ = [("n_scenes", C.c_int32), ("n_actors_total", C.c_int32), ("n_tl_total", C.c_int32)] + [
        (name, _P) for name in (
            "ego_state0", "ego_target_speed", "ego_tidx0", "len_ego_route", "num_vehicles", "ego_off", "rew_off",
            "actor_off", "tl_off", "ego_cx", "ego_cy", "ego_cyaw", "rew_rx", "rew_ry", "rew_cum", "act_kind",
            "act_state0", "act_tidx0", "act_cruise_px", "act_cruise_mps", "act_beh", "act_beh_p", "act_route_off",
            "act_raw_off", "act_cx", "act_cy", "act_cyaw", "act_raw_x", "act_raw_y", "tl_rect", "tl_color", "sg_mat")
    ]


class CbevStepOut(C.Structure):
    _fields_ = [("reward", _P), ("terminated", _P), ("truncated", _P), ("cause", _P), ("hero", _P), ("episode", _P)]


class CbevHostOut(C.Structure):
    _fields_ = [("reward", _P), ("terminated", _P), ("truncated", _P), ("cause", _P), ("episode", _P)]


class CbevSnapshotInfo(C.Structure):
    _fields_ = [("engine_token", C.c_uint64), ("pool_epoch", C.c_int32), ("retreat_slots", C.c_int32),
                ("row_bytes", C.c_int64), ("n_rows", C.c_int32), ("reserved", C.c_int32)]


class CbevLookaheadOut(C.Structure):
    _fields_ = [("ret", _P), ("reward", _P), ("steps", _P), ("terminated", _P), ("truncated", _P), ("cause", _P),
                ("hero", _P)]


class CbevLookaheadIo(C.Structure):
    _fields_ = [("src_info", C.POINTER(CbevSnapshotInfo)), ("src_rows", _P), ("roots", _P), ("obs", _P),
                ("obs_bytes", C.c_int64), ("leaf_rows", _P), ("leaf_bytes", C.c_int64),
                ("leaf_info", C.POINTER(CbevSnapshotInfo))]


class CbevError(RuntimeError):
    pass


class EnvSnapshot:
    """Rows taken by `Engine.snapshot`: `data` is a device uint8 tensor [n_rows, row_bytes] (one row per env, layout in
    csrc/engine.h), `info` the cbev_snapshot_info that ties the rows to the engine and pool epoch they were taken under.
    The rows are plain device memory: they can be cloned, sliced by row with `.data[i]` for inspection, and restored
    any number of times into any env of the same engine."""

    def __init__(self, buf, info):
        self._buf = buf  # storage, possibly more rows than the last snapshot used (`out=` reuse)
        self.info = info

    @property
    def data(self):
        return self._buf[: self.info.n_rows]

    @property
    def n_rows(self) -> int:
        return int(self.info.n_rows)

    @property
    def row_bytes(self) -> int:
        return int(self.info.row_bytes)

    def header(self):
        """int32 [n_rows, 3] device tensor: scene, episode, done of every row."""
        import torch

        return self.data[:, :12].contiguous().view(torch.int32)

    def __len__(self):
        return self.n_rows


class Lookahead:
    """Result of `Engine.lookahead`, device tensors over B branches: `ret` float64 [B] (discounted return, summed in
    step order), `steps` int32 [B] (steps taken, 0 when the root's last step was terminal), `terminated` / `truncated`
    bool [B] and `cause` uint8 [B] of the last step taken, and when asked for, `reward` float64 [H, B] (0.0 after a
    branch's last step), `hero` float64 [B, len(HERO_FIELDS)] (the hero block after the last step taken), and `obs`,
    the observation at each branch's leaf: the window [B, *Engine.obs().shape[1:]] in the ring's dtype, or with a
    fusion mode the fused window in the shape and dtype of `Engine.fuse(mode)`.  `window` is the raw leaf window
    (`obs` itself without fusion).  `leaf`, when asked for, is an `EnvSnapshot` of B rows: branch b's leaf state,
    which `Engine.restore` restores and `Engine.lookahead(source=...)` continues."""

    def __init__(self, ret, steps, terminated, truncated, cause, reward=None, hero=None, obs=None, window=None,
                 leaf=None):
        self.ret, self.steps, self.terminated, self.truncated, self.cause = ret, steps, terminated, truncated, cause
        self.reward, self.hero = reward, hero
        self.obs, self.window = obs, window
        self.leaf = leaf

    @property
    def n_branches(self) -> int:
        return int(self.ret.numel())

    @property
    def horizon(self):
        return None if self.reward is None else int(self.reward.shape[0])


_lib = None


def load_library(build_if_missing: bool = True):
    """dlopen libcbev.so; raises if it cannot be built/loaded (no silent fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH) or _build.needs_build():
        # a library older than csrc/ or include/cbev.h would run stale kernels behind an unchanged ABI
        if not build_if_missing:
            raise CbevError(f"{LIB_PATH} is missing or older than its sources; run `python -m carlabev_env_b200.build`")
        _build.build()
    lib = C.CDLL(LIB_PATH)
    lib.cbev_last_error.restype = C.c_char_p
    lib.cbev_frame_bytes.restype = C.c_int64
    lib.cbev_launch_count.restype = C.c_int64
    lib.cbev_frame_bytes.argtypes = [_P]
    lib.cbev_launch_count.argtypes = [_P]
    lib.cbev_create.argtypes = [C.POINTER(CbevConfig), C.POINTER(_P)]
    lib.cbev_destroy.argtypes = [_P]
    lib.cbev_upload_map.argtypes = [_P, _P, C.c_int32, C.c_int32]
    lib.cbev_upload_scene_pool.argtypes = [_P, C.POINTER(CbevPoolDesc)]
    lib.cbev_bind_obs_ring.argtypes = [_P, _P, C.c_int64]
    lib.cbev_reset.argtypes = [_P, _P, _P, _P]
    lib.cbev_step.argtypes = [_P, _P, C.POINTER(CbevStepOut), _P]
    lib.cbev_step_host.argtypes = [_P, _P, _P, _P, _P, _P]
    lib.cbev_step_host_ex.argtypes = [_P, _P, C.POINTER(CbevStepOut), C.POINTER(CbevHostOut), _P]
    lib.cbev_step_ex.argtypes = [_P, _P, C.POINTER(CbevStepOut), C.POINTER(CbevHostOut), _P]
    lib.cbev_invalidate.argtypes = [_P]
    lib.cbev_generate_scenes.argtypes = [_P, C.c_int32, _P, _P, _P, _P, _P]
    lib.cbev_pool_counts.argtypes = [_P, _P]
    lib.cbev_read_scene_pool.argtypes = [_P, C.POINTER(CbevPoolDesc)]
    lib.cbev_wait_host_outputs.argtypes = [_P]
    lib.cbev_set_state.argtypes = [_P, _P, _P]
    lib.cbev_profile_read_ex.argtypes = [_P, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double),
                                         C.POINTER(C.c_int64)]
    lib.cbev_obs_head.argtypes = [_P, C.POINTER(C.c_int32)]
    lib.cbev_get_state.argtypes = [_P, _P, _P]
    lib.cbev_set_ego_state.argtypes = [_P, _P]
    lib.cbev_copy_fov.argtypes = [_P, _P, _P]
    lib.cbev_keep_fov.argtypes = [_P, C.c_int32]
    lib.cbev_debug_read_trace.argtypes = [_P, _P]
    lib.cbev_upload_fov_mask.argtypes = [_P, _P]
    lib.cbev_fuse.argtypes = [_P, C.c_int32, _P, _P]
    lib.cbev_set_debug_flags.argtypes = [_P, C.c_int32]
    lib.cbev_set_action_repeat.argtypes = [_P, C.c_int32]
    lib.cbev_read_stats.argtypes = [_P, _P, C.c_int32, _P]
    lib.cbev_profile_enable.argtypes = [_P, C.c_int32]
    lib.cbev_profile_read.argtypes = [_P, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int64)]
    lib.cbev_abi_sizes.argtypes = [C.POINTER(C.c_int32)] * 3
    lib.cbev_snapshot_row_bytes.restype = C.c_int64
    lib.cbev_snapshot_row_bytes.argtypes = [_P]
    lib.cbev_snapshot.argtypes = [_P, _P, C.c_int32, _P, C.c_int64, C.POINTER(CbevSnapshotInfo), _P]
    lib.cbev_restore.argtypes = [_P, C.POINTER(CbevSnapshotInfo), _P, _P, _P, C.c_int32, _P]
    lib.cbev_lookahead.argtypes = [_P, _P, C.c_int32, C.c_int32, _P, C.c_double, C.POINTER(CbevLookaheadOut), _P]
    lib.cbev_lookahead_obs.argtypes = [_P, _P, C.c_int32, C.c_int32, _P, C.c_double, C.POINTER(CbevLookaheadOut), _P,
                                       C.c_int64, _P]
    lib.cbev_fuse_windows.argtypes = [_P, C.c_int32, _P, C.c_int32, _P, _P]
    lib.cbev_lookahead_ex.argtypes = [_P, C.POINTER(CbevLookaheadIo), C.c_int32, C.c_int32, _P, C.c_double,
                                      C.POINTER(CbevLookaheadOut), _P]
    sizes = [C.c_int32(), C.c_int32(), C.c_int32()]
    lib.cbev_abi_sizes(*[C.byref(v) for v in sizes])
    expect = (C.sizeof(CbevConfig), C.sizeof(CbevPoolDesc), C.sizeof(CbevStepOut))
    if tuple(v.value for v in sizes) != expect:
        raise CbevError(f"ABI mismatch between include/cbev.h and engine.py: {[v.value for v in sizes]} vs {expect}")
    _lib = lib
    return lib


def _check(lib, rc):
    if rc != 0:
        raise CbevError(f"cbev error {rc}: {lib.cbev_last_error().decode()}")


def savgol_operators() -> np.ndarray:
    """Linear operators of control/utils.py:smooth_and_compute's savgol stage for n-point routes,
    n <= SG_MAX (window 11 -> adapted, polyorder 3 -> adapted): sg[n] @ ax == smoothed ax."""
    from scipy.signal import savgol_filter

    sg = np.zeros((SG_MAX + 1, SG_MAX, SG_MAX), dtype=np.float64)
    for n in range(2, SG_MAX + 1):
        window = 11
        if window > n:
            window = n if n % 2 == 1 else n - 1
        if window < 3:
            window = 3
        poly = min(3, window - 1)
        if n >= window:
            m = savgol_filter(np.eye(n), window_length=window, polyorder=poly, axis=0)
        else:
            m = np.eye(n)
        sg[n, :n, :n] = m
    return sg


class Engine:
    """One engine = one GPU = one shard of environments."""

    def __init__(self, num_envs, *, obs_mode=OBS_SEMANTIC, mask_mode="6-class", frame_stack=4, ring_slots=None,
                 action_mode=ACTION_DISCRETE, discrete_table=None, reward_mode=REWARD_CARL, reward_params=None,
                 autoreset=AUTORESET_DISABLED, anchor=(0.5, 0.5), max_actors=0, seed=0, device=None,
                 ring_budget_bytes=None, size=128, obs_size=(96, 96), trajectory_steps=1024, mask_dtype="float32"):
        """`mask_dtype="uint8"` (obs_mode=OBS_SEMANTIC only) keeps the semantic masks as 0 / 1 bytes instead of float32:
        the same values, a quarter of the ring and of the raster kernel's stores (an extension beyond the reference)."""
        import torch

        if obs_mode not in (OBS_SEMANTIC, OBS_GRAY, OBS_RGB):
            raise ValueError(f"obs_mode must be OBS_SEMANTIC, OBS_GRAY or OBS_RGB, got {obs_mode!r} "
                             "(uint8 semantic masks are selected with mask_dtype='uint8')")
        if mask_dtype not in MASK_DTYPES:
            raise ValueError(f"mask_dtype must be one of {MASK_DTYPES}, got {mask_dtype!r}")
        if mask_dtype == "uint8" and obs_mode != OBS_SEMANTIC:
            raise ValueError("mask_dtype='uint8' applies to the semantic masks only (obs_mode=OBS_SEMANTIC)")
        if not torch.cuda.is_available():
            raise CbevError("carlabev_env_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.torch = torch
        self.lib = load_library()
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        torch.cuda.set_device(self.device)
        self.N = int(num_envs)
        self.obs_mode = obs_mode
        self.mask_mode = mask_mode
        self.mask_dtype = mask_dtype
        self.channels = MASK_CHANNELS[mask_mode] if obs_mode == OBS_SEMANTIC else 1
        self.F = 1 if obs_mode == OBS_RGB else int(frame_stack)
        self.size = int(size)
        self.obs_hw = tuple(obs_size)
        if obs_mode == OBS_SEMANTIC:
            frame = self.channels * obs_size[0] * obs_size[1] * (1 if mask_dtype == "uint8" else 4)
        elif obs_mode == OBS_GRAY:
            frame = obs_size[0] * obs_size[1]
        else:
            frame = size * size * 3
        if ring_slots is None:
            if self.F == 1:
                ring_slots = 1
            else:
                if ring_budget_bytes is None:
                    free, _ = torch.cuda.mem_get_info(self.device)
                    ring_budget_bytes = int(free * 0.35)
                # L >= 2F: the previous observation window stays intact for one more step (a caller holding both
                # `obs` and `next_obs` -- replay buffers, GAE bootstrap -- reads two valid windows); with the minimum
                # L = 2F - 1 the next head or mirror write lands inside the previous window
                ring_slots = max(2 * self.F, min(64, ring_budget_bytes // max(1, self.N * frame)))
        self.L = int(ring_slots)
        cfg = CbevConfig()
        cfg.num_envs = self.N
        cfg.fov_size = size
        cfg.anchor_x_frac, cfg.anchor_y_frac = float(anchor[0]), float(anchor[1])
        cfg.obs_h, cfg.obs_w = int(obs_size[0]), int(obs_size[1])
        cfg.obs_mode = OBS_SEMANTIC_U8 if mask_dtype == "uint8" else obs_mode
        cfg.mask_mode = MASK_MODES[mask_mode]
        cfg.frame_stack = self.F
        cfg.ring_slots = self.L
        cfg.action_mode = action_mode
        table = np.zeros((16, 3), dtype=np.float32)
        if action_mode == ACTION_DISCRETE:
            dt = np.asarray(discrete_table, dtype=np.float32).reshape(-1, 3)
            table[: len(dt)] = dt
            cfg.n_discrete = len(dt)
        for i, v in enumerate(table.ravel()):
            cfg.discrete_table[i] = float(v)
        cfg.reward_mode = reward_mode
        cfg.autoreset = autoreset
        cfg.max_actors = int(max_actors)
        cfg.trajectory_steps = int(trajectory_steps)
        params = dict(CARL_DEFAULTS)
        params.update(SHAPING_DEFAULTS)
        fixed = {"zero_speed_reward_offroad": True, "zero_progress_reward_offroad": True}  # what the kernels implement
        for k, v in (reward_params or {}).items():
            if k in params:
                params[k] = v
            elif k in fixed:
                if bool(v) != fixed[k]:
                    raise CbevError(f"reward parameter {k}={v!r} is not implemented (the engine computes {k}={fixed[k]})")
            else:
                raise CbevError(f"unknown reward parameter {k!r}; known: {sorted(params) + sorted(fixed)}")
        for k, v in params.items():
            setattr(cfg, k, v)
        cfg.seed = int(seed) & (2**64 - 1)
        self.cfg = cfg
        self.action_mode = action_mode
        self.handle = _P()
        _check(self.lib, self.lib.cbev_create(C.byref(cfg), C.byref(self.handle)))
        self.frame_bytes = int(self.lib.cbev_frame_bytes(self.handle))
        assert self.frame_bytes == frame
        # caller-owned buffers
        dev = self.device
        self.ring = torch.empty(self.N * self.L * frame, dtype=torch.uint8, device=dev)
        _check(self.lib, self.lib.cbev_bind_obs_ring(self.handle, self.ring.data_ptr(), self.ring.numel()))
        # reward f64[N] | terminated u8[N] | truncated u8[N] back to back: one D2H copy brings all three to the host
        self._rtt = torch.zeros(self.N * 10, dtype=torch.uint8, device=dev)
        self.reward = self._rtt[: self.N * 8].view(torch.float64)
        self.terminated = self._rtt[self.N * 8: self.N * 9]
        self.truncated = self._rtt[self.N * 9:]
        self._host = None  # pinned mirrors, allocated by the first step_host_full
        self.cause = torch.zeros(self.N, dtype=torch.uint8, device=dev)
        self.hero = torch.zeros(self.N, len(HERO_FIELDS), dtype=torch.float64, device=dev)
        self.episode = torch.zeros(self.N, len(EPISODE_FIELDS), dtype=torch.float64, device=dev)
        self.stats_buf = torch.zeros(STATS_FIELDS, dtype=torch.float64, device=dev)
        self._out = CbevStepOut(self.reward.data_ptr(), self.terminated.data_ptr(), self.truncated.data_ptr(),
                                self.cause.data_ptr(), self.hero.data_ptr(), self.episode.data_ptr())
        self._keep = []
        self.n_scenes = 0
        self._action_repeat = 1

    # ------------------------------------------------------------------ uploads
    def upload_map(self, cls_map: np.ndarray):
        m = np.ascontiguousarray(cls_map, dtype=np.uint8)
        _check(self.lib, self.lib.cbev_upload_map(self.handle, m.ctypes.data, m.shape[1], m.shape[0]))
        self.map_hw = m.shape

    def upload_pool(self, packed: dict):
        """packed = carlabev_env_b200.pool.pack_pool(scenes)."""
        d = CbevPoolDesc()
        keep = []

        def arr(key, dtype):
            a = np.ascontiguousarray(packed[key], dtype=dtype)
            keep.append(a)
            return a.ctypes.data if a.size else None

        d.n_scenes = int(packed["n_scenes"])
        d.n_actors_total = int(len(packed["act_kind"]))
        d.n_tl_total = int(len(packed["tl_color"]))
        for key, dt in (("ego_state0", np.float64), ("ego_target_speed", np.float64), ("ego_tidx0", np.int32),
                        ("len_ego_route", np.float64), ("num_vehicles", np.int32), ("ego_off", np.int32),
                        ("rew_off", np.int32), ("actor_off", np.int32), ("tl_off", np.int32), ("ego_cx", np.float64),
                        ("ego_cy", np.float64), ("ego_cyaw", np.float64), ("rew_rx", np.int32), ("rew_ry", np.int32),
                        ("act_kind", np.uint8), ("act_state0", np.float64), ("act_tidx0", np.int32),
                        ("act_cruise_px", np.float64), ("act_cruise_mps", np.float64), ("act_beh", np.uint8),
                        ("act_beh_p", np.float64), ("act_route_off", np.int32), ("act_raw_off", np.int32),
                        ("act_cx", np.float64), ("act_cy", np.float64), ("act_cyaw", np.float64),
                        ("act_raw_x", np.float64), ("act_raw_y", np.float64), ("tl_rect", np.int32),
                        ("tl_color", np.uint8)):
            setattr(d, key, arr(key, dt))
        # cumulative reward-route lengths exactly as carl_reward_fn.py:20-26 computes them (np.hypot of int deltas)
        rx, ry, off = packed["rew_rx"], packed["rew_ry"], packed["rew_off"]
        cum = np.zeros(len(rx), dtype=np.float64)
        for s in range(d.n_scenes):
            lo, hi = int(off[s]), int(off[s + 1])
            acc = 0.0
            for i in range(lo + 1, hi):
                acc = acc + np.hypot(rx[i] - rx[i - 1], ry[i] - ry[i - 1])
                cum[i] = acc
        keep.append(cum)
        d.rew_cum = cum.ctypes.data if cum.size else None
        sg = savgol_operators()
        keep.append(sg)
        d.sg_mat = sg.ctypes.data
        _check(self.lib, self.lib.cbev_upload_scene_pool(self.handle, C.byref(d)))
        self.n_scenes = d.n_scenes

    def generate_scripted_pool(self, kinds, levels, seeds):
        """Row f2: generate lead_brake / jaywalk scenes ON THE DEVICE from (kind, level, scene_seed) and make them the
        resident pool (cbev_generate_scenes).  kinds: "lead_brake" | "jaywalk" (or 1 | 2).  Returns the number of
        samples every scene needed (the reference's reset retry loop)."""
        ids = {"lead_brake": 1, "jaywalk": 2}
        k = np.ascontiguousarray([ids.get(v, v) for v in kinds], dtype=np.uint8)
        lv = np.ascontiguousarray(levels, dtype=np.int32)
        sd = np.ascontiguousarray(seeds, dtype=np.int64)
        assert len(k) == len(lv) == len(sd)
        sg = np.ascontiguousarray(savgol_operators())
        att = np.zeros(len(k), dtype=np.int32)
        _check(self.lib, self.lib.cbev_generate_scenes(self.handle, len(k), k.ctypes.data, lv.ctypes.data, sd.ctypes.data,
                                                       sg.ctypes.data, att.ctypes.data))
        self.n_scenes = len(k)
        return att

    def read_pool(self) -> dict:
        """The resident pool read back into host arrays (keys of pool.pack_pool that live on the device)."""
        c = np.zeros(8, dtype=np.int32)
        _check(self.lib, self.lib.cbev_pool_counts(self.handle, c.ctypes.data))
        n, na, nr, nq, npts, nw, ntl = (int(v) for v in c[:7])
        spec = (("ego_state0", np.float64, n * 4), ("ego_target_speed", np.float64, n), ("ego_tidx0", np.int32, n),
                ("len_ego_route", np.float64, n), ("num_vehicles", np.int32, n), ("ego_off", np.int32, n + 1),
                ("rew_off", np.int32, n + 1), ("actor_off", np.int32, n + 1), ("tl_off", np.int32, n + 1),
                ("ego_cx", np.float64, nr), ("ego_cy", np.float64, nr), ("ego_cyaw", np.float64, nr),
                ("rew_rx", np.int32, nq), ("rew_ry", np.int32, nq), ("rew_cum", np.float64, nq),
                ("act_kind", np.uint8, na), ("act_state0", np.float64, na * 4), ("act_tidx0", np.int32, na),
                ("act_cruise_px", np.float64, na), ("act_cruise_mps", np.float64, na), ("act_beh", np.uint8, na),
                ("act_beh_p", np.float64, na * 4), ("act_route_off", np.int32, na + 1), ("act_raw_off", np.int32, na + 1),
                ("act_cx", np.float64, npts), ("act_cy", np.float64, npts), ("act_cyaw", np.float64, npts),
                ("act_raw_x", np.float64, nw), ("act_raw_y", np.float64, nw), ("tl_rect", np.int32, ntl * 4),
                ("tl_color", np.uint8, ntl))
        d = CbevPoolDesc()
        out = {"n_scenes": n}
        for key, dt, cnt in spec:
            a = np.zeros(max(cnt, 1), dtype=dt)
            out[key] = a[:cnt]
            setattr(d, key, a.ctypes.data)
        _check(self.lib, self.lib.cbev_read_scene_pool(self.handle, C.byref(d)))
        out["ego_state0"] = out["ego_state0"].reshape(n, 4)
        out["act_state0"] = out["act_state0"].reshape(na, 4)
        out["act_beh_p"] = out["act_beh_p"].reshape(na, 4)
        out["tl_rect"] = out["tl_rect"].reshape(ntl, 4)
        return out

    # ------------------------------------------------------------------ stepping
    def _stream(self):
        return self.torch.cuda.current_stream(self.device).cuda_stream

    def reset(self, scene_ids, mask=None):
        t = self.torch
        ids = t.as_tensor(scene_ids, dtype=t.int32, device=self.device).contiguous()
        m = None
        if mask is not None:
            m = t.as_tensor(mask, device=self.device).to(t.uint8).contiguous()
        _check(self.lib, self.lib.cbev_reset(self.handle, None if m is None else m.data_ptr(), ids.data_ptr(),
                                             self._stream()))
        self._keep = [ids, m]
        return self.obs()

    @property
    def action_repeat(self) -> int:
        """Simulator steps per step call (`set_action_repeat`)."""
        return self._action_repeat

    def set_action_repeat(self, k: int):
        """Make every later step call one agent step of up to `k` simulator steps with the same action (1 <= k <= 64,
        an extension beyond the reference): an env stops at its first terminal sub-step, the reward is the sub-step
        rewards summed in order, the flags, cause, hero and episode blocks are those of the last sub-step, and one frame
        is rendered per call.  Reset, snapshot / restore and lookahead are unaffected; see cbev_set_action_repeat."""
        if isinstance(k, bool) or int(k) != k or not 1 <= int(k) <= MAX_ACTION_REPEAT:
            raise ValueError(f"action repeat must be an integer in [1, {MAX_ACTION_REPEAT}], got {k!r}")
        _check(self.lib, self.lib.cbev_set_action_repeat(self.handle, int(k)))
        self._action_repeat = int(k)

    def step(self, actions):
        """actions: device tensor int64[N] (discrete) or float32[N,3] (continuous)."""
        _check(self.lib, self.lib.cbev_step(self.handle, actions.data_ptr(), C.byref(self._out), self._stream()))

    def step_host(self, actions_host, reward_host, term_host, trunc_host):
        """Pinned host tensors in / out (the e2e path of bench.py)."""
        _check(self.lib, self.lib.cbev_step_host(self.handle, actions_host.data_ptr(), reward_host.data_ptr(),
                                                 term_host.data_ptr(), trunc_host.data_ptr(), self._stream()))

    def step_host_full(self, actions, episode=True):
        """Pinned host actions (or a CUDA tensor) in; reward / terminated / truncated (and the episode block) come back into pinned host
        mirrors (`host_reward`, `host_terminated`, `host_truncated`, `host_episode`) through D2H copies that overlap
        the raster kernel.  All device outputs (hero, cause, episode, ...) are written as in `step`.  Call
        `wait_host_outputs()` before reading the mirrors."""
        t = self.torch
        if self._host is None:
            blk = t.zeros(self.N * 10, dtype=t.uint8).pin_memory()
            self.host_reward = blk[: self.N * 8].view(t.float64)
            self.host_terminated = blk[self.N * 8: self.N * 9]
            self.host_truncated = blk[self.N * 9:]
            self.host_episode = t.zeros(self.N, len(EPISODE_FIELDS), dtype=t.float64).pin_memory()
            self._host = CbevHostOut(self.host_reward.data_ptr(), self.host_terminated.data_ptr(),
                                     self.host_truncated.data_ptr(), None, self.host_episode.data_ptr())
            self._host_noep = CbevHostOut(self.host_reward.data_ptr(), self.host_terminated.data_ptr(),
                                          self.host_truncated.data_ptr(), None, None)
            self._host_blk = blk
        fn = self.lib.cbev_step_ex if actions.is_cuda else self.lib.cbev_step_host_ex
        _check(self.lib, fn(self.handle, actions.data_ptr(), C.byref(self._out),
                            C.byref(self._host if episode else self._host_noep), self._stream()))

    def invalidate(self):
        """Every env must be reset before the next step (after the pool was replaced by an unrelated one)."""
        _check(self.lib, self.lib.cbev_invalidate(self.handle))

    def wait_host_outputs(self):
        """Block until the host copies of the last step_host / step_host_full have landed (the raster kernel of that
        step may still be running)."""
        _check(self.lib, self.lib.cbev_wait_host_outputs(self.handle))

    @property
    def head(self) -> int:
        h = C.c_int32(-1)
        _check(self.lib, self.lib.cbev_obs_head(self.handle, C.byref(h)))
        return h.value

    def obs(self):
        """Zero-copy view of the current observation window in the ring (semantic masks: float32, or uint8 with
        mask_dtype="uint8")."""
        t = self.torch
        head, F, L, N = self.head, self.F, self.L, self.N
        if self.obs_mode == OBS_SEMANTIC:
            ring = self.ring if self.mask_dtype == "uint8" else self.ring.view(t.float32)
            ring = ring.view(N, L, self.channels, *self.obs_hw)
            return ring[:, head - F + 1: head + 1].view(N, F * self.channels, *self.obs_hw)
        if self.obs_mode == OBS_GRAY:
            ring = self.ring.view(N, L, *self.obs_hw)
            return ring[:, head - F + 1: head + 1]
        return self.ring.view(N, self.size, self.size, 3)

    def upload_fov_mask(self, mask):
        """mask: uint8 [S, S], non-zero = painted black (fov_masked); None removes it."""
        if mask is None:
            _check(self.lib, self.lib.cbev_upload_fov_mask(self.handle, None))
            return
        m = np.ascontiguousarray(mask, dtype=np.uint8)
        assert m.shape == (self.size, self.size)
        _check(self.lib, self.lib.cbev_upload_fov_mask(self.handle, m.ctypes.data))

    def fuse(self, mode: str):
        """Temporal fusion of the current window: 'vehicle_temporal' -> [N, C+2, h, w] in the masks' dtype,
        'vehicle_weighted' -> float32 [N, C, h, w] (its values are not 0 / 1)."""
        code = FUSE_MODES[mode]
        t = self.torch
        key = ("fuse", code)
        buf = getattr(self, "_fuse_buf", {}).get(key)
        if buf is None:
            buf = t.empty(self.N, *self._fused_shape(code), dtype=self._fused_dtype(code), device=self.device)
            self._fuse_buf = {**getattr(self, "_fuse_buf", {}), key: buf}
        _check(self.lib, self.lib.cbev_fuse(self.handle, code, buf.data_ptr(), self._stream()))
        return buf

    def _fused_shape(self, code):
        return (self.channels + 2 if code == 1 else self.channels, *self.obs_hw)

    def _fused_dtype(self, code):
        t = self.torch
        return t.uint8 if code == 1 and self.mask_dtype == "uint8" else t.float32

    def _window_shape(self):
        """Per-env shape of `obs()`: [F*C, h, w] (semantic), [F, h, w] (gray), [S, S, 3] (raw RGB)."""
        if self.obs_mode == OBS_SEMANTIC:
            return (self.F * self.channels, *self.obs_hw)
        if self.obs_mode == OBS_GRAY:
            return (self.F, *self.obs_hw)
        return (self.size, self.size, 3)

    def _window_dtype(self):
        t = self.torch
        return t.float32 if self.obs_mode == OBS_SEMANTIC and self.mask_dtype != "uint8" else t.uint8

    # ------------------------------------------------------------------ snapshot / restore
    @property
    def snapshot_row_bytes(self) -> int:
        """Bytes of one snapshot row at the pool's current number of retreat slots."""
        return int(self.lib.cbev_snapshot_row_bytes(self.handle))

    def _index(self, idx, bound, what, unique):
        """(device int32 tensor, length) of an index argument.  An int32 CUDA tensor is used as it is (trusted: the
        kernels skip out-of-range entries); anything else is a host array, checked for range (and duplicates when
        `unique`) and sent with a stream-ordered copy from pinned memory -- neither path synchronises."""
        t = self.torch
        if isinstance(idx, t.Tensor) and idx.is_cuda:
            if idx.dtype != t.int32 or idx.dim() != 1 or idx.device != self.device:
                raise ValueError(f"{what}: a CUDA index tensor must be 1-D int32 on {self.device}")
            return idx.contiguous(), int(idx.numel())
        a = np.asarray(idx.numpy() if isinstance(idx, t.Tensor) else idx)
        if a.ndim != 1 or a.size == 0 or not np.issubdtype(a.dtype, np.integer):
            raise ValueError(f"{what} must be a non-empty 1-D integer array")
        if a.min() < 0 or a.max() >= bound:
            raise ValueError(f"{what} must lie in [0, {bound}), got [{a.min()}, {a.max()}]")
        if unique and len(np.unique(a)) != a.size:
            raise ValueError(f"{what} names an env more than once")
        host = t.from_numpy(a.astype(np.int32)).pin_memory()
        return host.to(self.device, non_blocking=True), int(a.size)

    def snapshot(self, env_ids=None, out=None) -> EnvSnapshot:
        """Copy the whole state of envs `env_ids` (default: all, row i = env i) into snapshot rows, on the device and in
        stream order.  `out=` reuses an earlier snapshot's storage (and returns that object), so a planning loop does
        not allocate."""
        t = self.torch
        ids, n = (None, self.N) if env_ids is None else self._index(env_ids, self.N, "env_ids", unique=False)
        rb = self.snapshot_row_bytes
        if out is None:
            buf = t.empty(n, rb, dtype=t.uint8, device=self.device)
        else:
            buf = out._buf
            if buf.device != self.device or buf.shape[1] != rb or buf.shape[0] < n:
                raise ValueError(f"out= holds {tuple(buf.shape)} rows x bytes on {buf.device}; this snapshot needs "
                                 f"({n}, {rb}) on {self.device}")
        info = CbevSnapshotInfo()
        _check(self.lib, self.lib.cbev_snapshot(self.handle, None if ids is None else ids.data_ptr(), n, buf.data_ptr(),
                                                buf.numel(), C.byref(info), self._stream()))
        self._keep_snap = ids
        if out is None:
            return EnvSnapshot(buf, info)
        out.info = info
        return out

    def restore(self, snap: EnvSnapshot, env_ids=None, rows=None):
        """Write row rows[i] of `snap` into env env_ids[i] (defaults: identity) and return the current observation.
        Restoring one row into several envs clones it; every env then continues bit-identically to the env the row
        was taken from, until its next device auto-reset (whose scene draw depends on the env index).  The window
        frames are rewritten in place: a zero-copy `obs()` view held for these envs changes."""
        if not isinstance(snap, EnvSnapshot):
            raise TypeError("restore() takes an EnvSnapshot returned by snapshot()")
        ids, ni = (None, None) if env_ids is None else self._index(env_ids, self.N, "env_ids", unique=True)
        rws, nr = (None, None) if rows is None else self._index(rows, snap.n_rows, "rows", unique=False)
        if ni is not None and nr is not None and ni != nr:
            raise ValueError(f"env_ids ({ni}) and rows ({nr}) must have the same length")
        n = ni if ni is not None else (nr if nr is not None else snap.n_rows)
        _check(self.lib, self.lib.cbev_restore(self.handle, C.byref(snap.info), snap._buf.data_ptr(),
                                               None if rws is None else rws.data_ptr(),
                                               None if ids is None else ids.data_ptr(), n, self._stream()))
        self._keep_snap = (ids, rws)
        return self.obs()

    # ------------------------------------------------------------------ lookahead
    def lookahead(self, actions, env_ids=None, gamma=1.0, rewards=False, hero=False, obs=False, fuse=None,
                  out=None, *, source=None, rows=None, leaf=False) -> Lookahead:
        """Roll B branches H steps ahead without rendering and return their rewards (planning: MPC, CEM, MCTS).
        Branch b starts from the current state of env `env_ids[b]` (default: env b) and takes `actions[t, b]` --
        a CUDA tensor, int64 [H, B] (discrete) or float32 [H, B, 3] (continuous) -- stopping after its first terminal
        step.  Rewards, flags, causes and hero blocks are bit-identical to stepping those envs with those actions, and
        the live envs, the observation ring, the episode statistics and the last step's outputs are left untouched.
        `env_ids` may repeat (a host array is range-checked, an int32 CUDA tensor is trusted); nothing synchronises.
        `rewards=True` / `hero=True` also return the per-step rewards and the final hero blocks.
        `obs=True` also renders each branch's leaf observation (`la.obs`, [B, *obs().shape[1:]]): byte-identical to
        `obs()` of an env cloned from the root and stepped with the branch's actions for `steps[b]` steps, the frames
        older than the branch's first step coming from the root's current window.  `fuse="vehicle_temporal"` or
        `"vehicle_weighted"` (semantic masks) returns that window fused as `fuse(mode)` would (`la.window` keeps the
        raw window).  `out=` reuses the storage of an earlier result of the same B (and H, with rewards; with the
        same obs / fuse buffers) and returns that object.
        `source=` (an `EnvSnapshot` of this engine and pool epoch) starts branch b from row `rows[b]` of it (default:
        row b) instead of a live env; every output is then what a call from an env restored from that row gives.
        `rows` may repeat (host arrays are range-checked, int32 CUDA tensors are trusted).  `leaf=True` also returns
        each branch's leaf state as snapshot row b of `la.leaf` (an `EnvSnapshot` of B rows): `restore` continues it
        in a live env and `lookahead(source=la.leaf)` continues it as a branch, both bit-identically.  Leaf rows carry
        their frames (one row is `snapshot_row_bytes`, about 885 KB with float32 masks and 222 KB with uint8 ones at
        96 x 96, F = 4), so `leaf=True` renders the leaf windows even without `obs=True`.  With `out=`, `la.leaf`'s
        storage is reused, or replaced when the row size has grown (a pool extension with more retreat slots)."""
        t = self.torch
        if not isinstance(actions, t.Tensor) or not actions.is_cuda or actions.device != self.device:
            raise ValueError(f"actions must be a CUDA tensor on {self.device}")
        if self.action_mode == ACTION_DISCRETE:
            if actions.dtype != t.int64 or actions.dim() != 2:
                raise ValueError(f"discrete actions must be int64 [H, B], got {actions.dtype} {tuple(actions.shape)}")
        elif actions.dtype != t.float32 or actions.dim() != 3 or actions.shape[2] != 3:
            raise ValueError(f"continuous actions must be float32 [H, B, 3], got {actions.dtype} {tuple(actions.shape)}")
        H, B = int(actions.shape[0]), int(actions.shape[1])
        if H < 1 or B < 1:
            raise ValueError(f"actions must hold at least one step of one branch, got shape {tuple(actions.shape)}")
        gamma = float(gamma)
        if not np.isfinite(gamma):
            raise ValueError(f"gamma must be finite, got {gamma}")
        if rows is not None and source is None:
            raise ValueError("rows= names rows of source=: it needs source=")
        if source is not None:
            if env_ids is not None:
                raise ValueError("env_ids= and source= are exclusive: the roots are live envs or rows of source")
            if not isinstance(source, EnvSnapshot):
                raise TypeError("source= takes an EnvSnapshot (snapshot() or a lookahead's leaf)")
            if source._buf.device != self.device:
                raise ValueError(f"source= rows are on {source._buf.device}, the engine on {self.device}")
        ids = None
        if source is not None and rows is not None:
            ids, n = self._index(rows, source.n_rows, "rows", unique=False)
            if n != B:
                raise ValueError(f"rows names {n} roots, actions have {B} branches")
        elif source is not None:
            if B > source.n_rows:
                raise ValueError(f"{B} branches without rows start from rows 0..{B - 1}, but source has "
                                 f"{source.n_rows}")
        elif env_ids is not None:
            ids, n = self._index(env_ids, self.N, "env_ids", unique=False)
            if n != B:
                raise ValueError(f"env_ids names {n} roots, actions have {B} branches")
        elif B > self.N:
            raise ValueError(f"{B} branches without env_ids start from envs 0..{B - 1}, but there are {self.N} envs")
        code = None
        if fuse is not None:
            if fuse not in FUSE_MODES:
                raise ValueError(f"fuse must be one of {sorted(FUSE_MODES)}, got {fuse!r}")
            if not obs:
                raise ValueError("fuse= fuses the leaf observation: it needs obs=True")
            if self.obs_mode != OBS_SEMANTIC:
                raise ValueError("fuse= requires obs_mode='bev_semantic'")
            code = FUSE_MODES[fuse]
        wshape, wdtype = (B, *self._window_shape()), self._window_dtype()
        fshape, fdtype = ((B, *self._fused_shape(code)), self._fused_dtype(code)) if code else (None, None)
        actions = actions.contiguous()
        if out is None:
            dev = self.device
            win = t.empty(wshape, dtype=wdtype, device=dev) if obs else None
            out = Lookahead(t.empty(B, dtype=t.float64, device=dev), t.empty(B, dtype=t.int32, device=dev),
                            t.empty(B, dtype=t.bool, device=dev), t.empty(B, dtype=t.bool, device=dev),
                            t.empty(B, dtype=t.uint8, device=dev),
                            t.empty(H, B, dtype=t.float64, device=dev) if rewards else None,
                            t.empty(B, len(HERO_FIELDS), dtype=t.float64, device=dev) if hero else None,
                            (t.empty(fshape, dtype=fdtype, device=dev) if code else win), win)
            if leaf:
                out.leaf = EnvSnapshot(t.empty(B, self.snapshot_row_bytes, dtype=t.uint8, device=dev),
                                       CbevSnapshotInfo())
        else:
            if not isinstance(out, Lookahead):
                raise TypeError("out= takes a Lookahead returned by lookahead()")
            if out.n_branches != B or out.ret.device != self.device:
                raise ValueError(f"out= holds {out.n_branches} branches on {out.ret.device}; this call has {B} on "
                                 f"{self.device}")
            if rewards and (out.reward is None or tuple(out.reward.shape) != (H, B)):
                raise ValueError(f"out= has no [{H}, {B}] reward buffer")
            if hero and out.hero is None:
                raise ValueError("out= has no hero buffer")
            if obs and (out.window is None or tuple(out.window.shape) != wshape or out.window.dtype != wdtype):
                raise ValueError(f"out= has no {wdtype} {list(wshape)} leaf-window buffer")
            if code and (out.obs is None or out.obs is out.window or tuple(out.obs.shape) != fshape
                         or out.obs.dtype != fdtype):
                raise ValueError(f"out= has no {fdtype} {list(fshape)} buffer for fuse={fuse!r}")
            if obs and not code:
                out.obs = out.window
            rb = self.snapshot_row_bytes
            if leaf and (out.leaf is None or out.leaf._buf.shape[1] != rb or out.leaf._buf.shape[0] < B):
                out.leaf = EnvSnapshot(t.empty(B, rb, dtype=t.uint8, device=self.device), CbevSnapshotInfo())
        o = CbevLookaheadOut(out.ret.data_ptr(), out.reward.data_ptr() if rewards else None, out.steps.data_ptr(),
                             out.terminated.data_ptr(), out.truncated.data_ptr(), out.cause.data_ptr(),
                             out.hero.data_ptr() if hero else None)
        roots = None if ids is None else ids.data_ptr()
        if source is not None or leaf:
            win = out.window if obs else None
            lf = out.leaf if leaf else None
            io = CbevLookaheadIo(C.pointer(source.info) if source is not None else None,
                                 source._buf.data_ptr() if source is not None else None, roots,
                                 win.data_ptr() if obs else None, win.numel() * win.element_size() if obs else 0,
                                 lf._buf.data_ptr() if leaf else None, lf._buf.numel() if leaf else 0,
                                 C.pointer(lf.info) if leaf else None)
            rc = self.lib.cbev_lookahead_ex(self.handle, C.byref(io), B, H, actions.data_ptr(), gamma, C.byref(o),
                                            self._stream())
            if rc != 0:
                msg = self.lib.cbev_last_error().decode()
                if "src rows" in msg:  # a foreign or stale source, refused from its info before any launch
                    raise ValueError(msg)
                _check(self.lib, rc)
            if code:
                _check(self.lib, self.lib.cbev_fuse_windows(self.handle, code, win.data_ptr(), B, out.obs.data_ptr(),
                                                            self._stream()))
            self._keep_look = (ids, actions, source)
            return out
        if obs:
            win = out.window
            _check(self.lib, self.lib.cbev_lookahead_obs(self.handle, roots, B, H, actions.data_ptr(), gamma,
                                                         C.byref(o), win.data_ptr(),
                                                         win.numel() * win.element_size(), self._stream()))
            if code:
                _check(self.lib, self.lib.cbev_fuse_windows(self.handle, code, win.data_ptr(), B, out.obs.data_ptr(),
                                                            self._stream()))
        else:
            _check(self.lib, self.lib.cbev_lookahead(self.handle, roots, B, H, actions.data_ptr(), gamma, C.byref(o),
                                                     self._stream()))
        self._keep_look = (ids, actions)
        return out

    def set_debug_flags(self, flags: int):
        _check(self.lib, self.lib.cbev_set_debug_flags(self.handle, int(flags)))

    def read_trace(self):
        """Per-CTA phase timestamps of the last raster launch, uint64 [N, 8] (set_debug_flags(4) first)."""
        out = np.zeros((self.N, 8), dtype=np.uint64)
        _check(self.lib, self.lib.cbev_debug_read_trace(self.handle, out.ctypes.data))
        return out

    def keep_fov(self, on=True):
        _check(self.lib, self.lib.cbev_keep_fov(self.handle, int(on)))

    def fov(self):
        """Last rendered palette-index frames, uint8 [N, S, S] (needs keep_fov(True) before the step)."""
        out = self.torch.empty(self.N, self.size, self.size, dtype=self.torch.uint8, device=self.device)
        _check(self.lib, self.lib.cbev_copy_fov(self.handle, out.data_ptr(), self._stream()))
        return out

    def get_state(self, max_actors=None):
        """(ego [N, 16], actors [N, max_actors, 8]) of cbev_get_state; the library always writes the engine's full
        actor capacity, the returned block is cut to `max_actors` columns."""
        cap = max(1, int(self.cfg.max_actors))
        ego = np.zeros((self.N, 16), dtype=np.float64)
        act = np.zeros((self.N, cap, 8), dtype=np.float64)
        _check(self.lib, self.lib.cbev_get_state(self.handle, ego.ctypes.data, act.ctypes.data))
        return ego, (act if max_actors is None else act[:, :max(1, max_actors)])

    def set_ego_state(self, ego):
        e = np.ascontiguousarray(ego, dtype=np.float64)
        _check(self.lib, self.lib.cbev_set_ego_state(self.handle, e.ctypes.data))

    def set_state(self, ego=None, actors=None):
        """Debug / parity: write back blocks in the layout of get_state (either may be None)."""
        e = None if ego is None else np.ascontiguousarray(ego, dtype=np.float64)
        a = None if actors is None else np.ascontiguousarray(actors, dtype=np.float64)
        if a is not None:
            assert a.shape == (self.N, max(1, int(self.cfg.max_actors)), 8), a.shape
        _check(self.lib, self.lib.cbev_set_state(self.handle, None if e is None else e.ctypes.data,
                                                 None if a is None else a.ctypes.data))

    def read_stats(self, reset=False):
        _check(self.lib, self.lib.cbev_read_stats(self.handle, self.stats_buf.data_ptr(), int(reset), self._stream()))
        return self.stats_buf

    def profile(self, on: bool):
        _check(self.lib, self.lib.cbev_profile_enable(self.handle, int(on)))

    def profile_read(self):
        """(move_ms, render_ms, judge_ms, steps) summed over the profiled steps since the last read; k_judge runs on
        the side stream concurrently with k_render."""
        a, b, c, n = C.c_double(), C.c_double(), C.c_double(), C.c_int64()
        _check(self.lib, self.lib.cbev_profile_read_ex(self.handle, C.byref(a), C.byref(b), C.byref(c), C.byref(n)))
        return a.value, b.value, c.value, n.value

    @property
    def launches(self) -> int:
        return int(self.lib.cbev_launch_count(self.handle))

    def close(self):
        if self.handle:
            self.torch.cuda.synchronize(self.device)
            self.lib.cbev_destroy(self.handle)
            self.handle = _P()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

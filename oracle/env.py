"""Oracle: single-env and vector-env front ends.  TEST INFRASTRUCTURE ONLY.

OracleEnv restates CarlaBEV.reset/step/render (envs/carlabev.py:96-249) plus the wrapper chain
of wrap_env (envs/__init__.py:40-90): ResizeObservation -> SemanticMaskWrapper | GrayscaleObservation
-> FrameStackObservation -> FlattenStackedFrames -> RecordEpisodeStatistics.
OracleVectorEnv restates gymnasium SyncVectorEnv with AutoresetMode.DISABLED (envs/__init__.py:116-119).
"""
from __future__ import annotations

from collections import deque

import numpy as np

from . import raster
from .sim import CAUSE_NAMES, DISCRETE9, DISCRETE13, SceneSim


def unpack_pool(npz):
    """Inverse of carlabev_env_b200.pool.pack_pool: dict of concatenated arrays -> list of scene dicts."""
    npz = {k: np.asarray(npz[k]) for k in (npz.files if hasattr(npz, "files") else npz.keys())}  # decompress once
    n = int(npz["n_scenes"])
    scenes = []
    per_scene = ["ego_state0", "ego_target_speed", "ego_tidx0", "route_length_m", "len_ego_route", "num_vehicles",
                 "kind", "level", "seed"]
    for i in range(n):
        s = {k: npz[k][i] for k in per_scene if k in npz}
        lo, hi = npz["ego_off"][i], npz["ego_off"][i + 1]
        for k in ("ego_cx", "ego_cy", "ego_cyaw"):
            s[k] = np.array(npz[k][lo:hi])
        lo, hi = npz["rew_off"][i], npz["rew_off"][i + 1]
        for k in ("rew_rx", "rew_ry"):
            s[k] = np.array(npz[k][lo:hi])
        a0, a1 = npz["actor_off"][i], npz["actor_off"][i + 1]
        for k in ("act_kind", "act_state0", "act_tidx0", "act_cruise_px", "act_cruise_mps", "act_beh", "act_beh_p"):
            s[k] = np.array(npz[k][a0:a1])
        ro = np.array(npz["act_route_off"][a0:a1 + 1])
        for k in ("act_cx", "act_cy", "act_cyaw"):
            s[k] = np.array(npz[k][ro[0]:ro[-1]])
        s["act_route_off"] = (ro - ro[0]).astype(np.int32)
        ro = np.array(npz["act_raw_off"][a0:a1 + 1])
        for k in ("act_raw_x", "act_raw_y"):
            s[k] = np.array(npz[k][ro[0]:ro[-1]])
        s["act_raw_off"] = (ro - ro[0]).astype(np.int32)
        t0, t1 = npz["tl_off"][i], npz["tl_off"][i + 1]
        s["tl_rect"] = np.array(npz["tl_rect"][t0:t1]).reshape(-1, 4)
        s["tl_color"] = np.array(npz["tl_color"][t0:t1])
        scenes.append(s)
    return scenes


class OracleEnv:
    def __init__(self, cls_map, *, obs_mode="bev_semantic", semantic_mask_ch="6-class", frame_stack=4,
                 obs_size=(96, 96), action_mode="discrete", action_profile="discrete9_v1", reward_mode="carl",
                 reward_params=None, anchor=(0.5, 0.5), size=128, fov_masked=False, temporal_fusion_mode="stack"):
        self.cls_map = np.ascontiguousarray(cls_map, dtype=np.uint8)
        self.geom = raster.FovGeometry(size, anchor[0], anchor[1])
        self.obs_mode = obs_mode
        self.fov_mask = raster.corner_mask(size, 0.5) if fov_masked else None
        self.fusion = temporal_fusion_mode
        self.mask_mode = semantic_mask_ch
        self.frame_stack = int(frame_stack)
        self.obs_size = tuple(obs_size)
        self.action_mode = action_mode
        self.table = DISCRETE13 if action_profile == "discrete13_v1" else DISCRETE9
        self.reward_mode = reward_mode
        self.reward_params = reward_params
        self.sim = None
        self.frames = deque(maxlen=self.frame_stack)
        self.episode = 0
        self.history = deque(maxlen=200)  # (cause, return) per finished episode, stats.py:100-125

    # -- observation pipeline ------------------------------------------------
    def render_index(self, reset_frame=False):
        s = self.sim
        theta = 0.0 if reset_frame else s.ego.yaw  # world.py:92-100: reset draws with _theta = 0 and no actors
        rects = raster.draw_list(s, with_actors=not reset_frame)
        return raster.render_fov(self.cls_map, self.geom, s.ego.x, s.ego.y, theta, rects, self.fov_mask)

    def _wrap_frame(self, idx_img):
        rgb = raster.fov_rgb(idx_img)
        self.last_rgb = rgb
        if self.obs_mode == "bev_raw":
            return rgb
        small = raster.resize_area(rgb, self.obs_size)
        if self.obs_mode == "bev_semantic":
            return raster.semantic_masks(small, self.mask_mode)
        return raster.grayscale(small)

    def _stacked(self):
        st = np.stack(list(self.frames))
        if self.obs_mode == "bev_semantic" and self.fusion == "vehicle_temporal":
            return raster.fuse_vehicle_temporal(st, self.mask_mode)
        if self.obs_mode == "bev_semantic" and self.fusion == "vehicle_weighted":
            return raster.fuse_vehicle_weighted(st, self.mask_mode)
        if self.obs_mode == "bev_semantic":
            return st.reshape(-1, *st.shape[2:]).astype(np.float32)  # FlattenStackedFrames
        return st

    # -- gym surface ------------------------------------------------------------
    def reset(self, scene):
        self.sim = SceneSim(scene, self.cls_map, self.geom.pad, self.reward_mode, self.reward_params, size=self.geom.size)
        self.ep_return = 0.0
        self.ep_len = 0
        frame = self._wrap_frame(self.render_index(reset_frame=True))
        self.frames.clear()
        for _ in range(self.frame_stack):
            self.frames.append(frame)
        return self._stacked()

    def push_frame(self):
        """Render the current state into the frame stack and return the stacked observation."""
        self.frames.append(self._wrap_frame(self.render_index()))
        return self._stacked()

    def step(self, action, render=True):
        """`render=False` leaves the frame stack alone and returns None as the observation: an agent step of action
        repeat K renders only its last simulator step (`push_frame` after it)."""
        s = self.sim
        gas, steer, brake = s.decode_action(action, self.action_mode, self.table)
        reward, terminated, truncated, cause = s.step(gas, steer, brake)
        obs = self.push_frame() if render else None
        self.ep_return += reward
        self.ep_len += 1
        info = {}
        if terminated:
            summ = s.episode_summary()
            hist = list(self.history)
            causes = [c for c, _ in hist]
            frac = lambda name: causes.count(name) / len(causes) if causes else 0.0  # noqa: E731
            summ.update(episode=self.episode, mean_reward=float(np.mean([r for _, r in hist])) if hist else 0.0,
                        success_rate=frac("success"), collision_rate=frac("collision"),
                        unfinished_rate=frac("off_road"), mean_ttc=0.0, mean_progress=0.0,
                        num_vehicles=int(s.scene["num_vehicles"]), len_ego_route=float(s.scene["len_ego_route"]))
            self.history.append((CAUSE_NAMES[s.ep_cause], summ["return"]))
            self.episode += 1
            s.stats_reset()
            info["episode_info"] = summ
            info["episode"] = {"r": self.ep_return, "l": self.ep_len}
        return obs, reward, terminated, truncated, info


class OracleVectorEnv:
    """Serial loop over OracleEnv with reset_mask semantics (gymnasium SyncVectorEnv, DISABLED autoreset)."""

    def __init__(self, num_envs, cls_map, **kw):
        self.envs = [OracleEnv(cls_map, **kw) for _ in range(num_envs)]
        self.num_envs = num_envs
        self._obs = [None] * num_envs

    def reset(self, scenes, reset_mask=None):
        for i, env in enumerate(self.envs):
            if reset_mask is None or reset_mask[i]:
                self._obs[i] = env.reset(scenes[i])
        return np.stack(self._obs)

    def step(self, actions):
        rew = np.zeros(self.num_envs, dtype=np.float64)
        term = np.zeros(self.num_envs, dtype=bool)
        trunc = np.zeros(self.num_envs, dtype=bool)
        infos = [None] * self.num_envs
        for i, env in enumerate(self.envs):
            self._obs[i], rew[i], term[i], trunc[i], infos[i] = env.step(actions[i])
        return np.stack(self._obs), rew, term, trunc, infos

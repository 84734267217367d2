"""Drop-in vectorised CarlaBEV environment on top of the CUDA engine.

Surface kept from the reference (`CarlaBEV.envs.make_env` -> gymnasium SyncVectorEnv of wrapped
CarlaBEV envs; envs/__init__.py:40-120, envs/carlabev.py:36-258):

    envs = make_env(cfg)                      # RunConfig | EnvConfig | legacy attribute bag
    envs.num_envs, envs.single_observation_space, envs.single_action_space
    obs, infos = envs.reset(seed=None, options={"scene": ..., "level": ..., "scene_seed": ...,
                                                "reset_mask": bool[N]})
    obs, rewards, terminations, truncations, infos = envs.step(actions)
    envs.close()

Differences that follow from the design (see DESIGN.md):
  * observations / rewards / flags are torch CUDA tensors (the step never leaves the GPU);
    `to_numpy=True` returns NumPy copies with the reference's dtypes.
  * `mask_dtype="uint8"` (bev_semantic only, an extension) returns the 0 / 1 masks as uint8 instead of float32.
  * `action_repeat=K` (an extension) makes each `step` K simulator steps with the same action, one rendered frame
    and the summed reward; `episode_info["length"]` counts simulator steps, `episode["l"]` agent steps.
  * scenes come from a host-generated, device-resident pool; `reset(options=...)` selects or
    extends it.  `autoreset="next_step"` turns on device auto-reset from that pool (gymnasium's NEXT_STEP), and
    `autoreset="same_step"` resets in the terminal step itself (gymnasium's SAME_STEP): `infos["final_obs"]` /
    `infos["final_info"]` then carry the terminal observation and the terminal keys.
  * `host_infos=False` (with device auto-reset) makes `step` fully asynchronous: no host synchronisation,
    terminal summaries stay in `infos["episode_block"]` (CBEV_E_* columns) on the device.
  * `infos` carries the reference's terminal keys (`episode_info`, `episode`) as dict-of-arrays
    with `_key` masks, plus the per-step `hero` comfort signals the reference documents
    (docs/control_and_actions.md:102) as a batched tensor.
"""
from __future__ import annotations

import os
import time

import numpy as np

from . import engine as E
from . import scenes as S
from .config import (SHAPING_DEFAULTS, RunConfig, get_action_profile_spec, get_reward_profile_spec,
                     validate_run_config)
from .pool import load_shipped_pool, pack_pool, shipped_pool_for
from .spaces import Box, Discrete

HERE = os.path.dirname(os.path.abspath(__file__))
_CAUSE_ARRAY = np.array(E.CAUSE_NAMES, dtype=object)


def load_town01_map(size: int = 128) -> np.ndarray:
    """Class map of Town01 at EnvConfig.size (64: 640 x 512, 128: 1280 x 1024, 256: 2560 x 2048 (rows x columns);
    0 non-drivable, 1 drivable, 2 sidewalk), derived from the reference's Town01-<size>-sem.png by
    oracle/gen_golden.py:dump_map (envs/utils.py:49-62)."""
    path = os.path.join(HERE, "assets", f"town01_{int(size)}_cls.npz")
    if not os.path.exists(path):
        raise ValueError(f"size={size}: no Town01 class map of that scale ships (64, 128, 256)")
    with np.load(path) as z:
        return np.ascontiguousarray(z["cls"], dtype=np.uint8)


def _vector_env_base():
    """gymnasium.vector.VectorEnv when gymnasium is importable (isinstance checks of downstream trainers then hold);
    the image this was built in has no gymnasium wheel, so a plain object otherwise."""
    try:
        from gymnasium.vector import VectorEnv

        return VectorEnv
    except Exception:  # noqa: BLE001
        return object


class CarlaBEVVectorEnv(_vector_env_base()):
    metadata = {"render_modes": ["rgb_array"], "render_fps": 60, "autoreset_mode": "Disabled"}

    def __init__(self, cfg: RunConfig, *, scenes=None, autoreset: str = "disabled", device=None, ring_slots=None,
                 ring_budget_bytes=None, to_numpy: bool = False, raw_rgb: bool = False, seed=None,
                 host_infos: bool = True, eval: bool = False, shard=None, mask_dtype: str = "float32",
                 action_repeat: int = 1):  # noqa: A002
        import torch

        if isinstance(action_repeat, bool) or int(action_repeat) != action_repeat \
                or not 1 <= int(action_repeat) <= E.MAX_ACTION_REPEAT:
            raise ValueError(f"action_repeat must be an integer in [1, {E.MAX_ACTION_REPEAT}], got {action_repeat!r}")

        self.torch = torch
        self.cfg = cfg
        env = cfg.env
        self.env_cfg = env
        self.fusion = env.temporal_fusion_mode if env.obs_mode == "bev_semantic" else "stack"
        if autoreset == "same_step":
            if getattr(cfg, "capture_video", False):
                raise ValueError("autoreset='same_step' does not support capture_video (the recorder follows the "
                                 "next_step auto-reset); use autoreset='next_step' to record")
            if self.fusion != "stack" and not host_infos:
                raise ValueError("autoreset='same_step' with temporal_fusion_mode needs host_infos=True: the final "
                                 "windows of the finished envs are fused by their indices on the host")
            try:
                from gymnasium.vector import AutoresetMode

                mode = AutoresetMode.SAME_STEP
            except Exception:  # noqa: BLE001
                mode = "SameStep"
            self.metadata = {**type(self).metadata, "autoreset_mode": mode}
        # shard = (rank, world_size): this process owns the contiguous env range [lo, hi) of cfg.num_envs
        # (distributed.shard_range); env i of the shard behaves like env lo + i of the unsharded VectorEnv
        self.env_offset = 0
        self.num_envs = int(cfg.num_envs)
        if shard is not None:
            from .distributed import shard_range

            lo, hi = shard_range(int(cfg.num_envs), int(shard[0]), int(shard[1]))
            self.env_offset, self.num_envs = lo, hi - lo
        self.to_numpy = to_numpy
        self.host_infos = host_infos or autoreset == "disabled"  # masked-reset bookkeeping needs the done flags
        self.autoreset = autoreset
        aspec = get_action_profile_spec(env.action_profile_id)
        rspec = get_reward_profile_spec(env.reward_profile_id)
        if env.obs_mode == "bev_semantic":
            obs_mode = E.OBS_SEMANTIC
        elif raw_rgb:
            obs_mode = E.OBS_RGB
        else:
            obs_mode = E.OBS_GRAY  # wrap_env: bev_rgb -> GrayscaleObservation (envs/__init__.py:70)
        self._scenes = list(scenes) if scenes is not None else []
        self._pool_is_user = scenes is not None  # reset() without a scene draws from a pool the caller passed in
        max_actors = max([len(s["act_kind"]) for s in self._scenes] + [env.max_vehicles + 2])
        params = dict(rspec["parameters"])
        if env.reward_mode == "shaping":
            params.setdefault("max_actions", SHAPING_DEFAULTS["max_actions"])  # cfg.max_actions is never passed
        self.engine = E.Engine(
            self.num_envs, obs_mode=obs_mode, mask_mode=env.semantic_mask_ch, frame_stack=env.frame_stack,
            ring_slots=ring_slots, ring_budget_bytes=ring_budget_bytes,
            action_mode=E.ACTION_DISCRETE if env.action_mode == "discrete" else E.ACTION_CONTINUOUS,
            discrete_table=aspec.get("discrete_actions"),
            reward_mode=E.REWARD_CARL if env.reward_mode == "carl" else E.REWARD_SHAPING, reward_params=params,
            autoreset={"next_step": E.AUTORESET_NEXT_STEP, "same_step": E.AUTORESET_SAME_STEP}.get(
                autoreset, E.AUTORESET_DISABLED),
            anchor=(env.ego_anchor_x_frac, env.ego_anchor_y_frac), max_actors=max_actors,
            seed=(cfg.seed if seed is None else seed) + (int(shard[0]) if shard is not None else 0),  # auto-reset draws
            device=device, size=env.size, obs_size=env.obs_size, mask_dtype=mask_dtype)
        # a keyword, not an EnvConfig field (EnvConfig mirrors the reference's schema), fixed for the env's lifetime
        self.action_repeat = int(action_repeat)
        if self.action_repeat > 1:
            self.engine.set_action_repeat(self.action_repeat)
        self.device = self.engine.device
        self.cls_map = load_town01_map(env.size)
        self.engine.upload_map(self.cls_map)
        self.pad = self._crop_size(env)
        if env.fov_masked:  # FovRenderSpec(mask_fov=True), envs/world.py:39-46
            from .fovmask import corner_mask

            self.engine.upload_fov_mask(corner_mask(env.size, 0.5))
        if self._scenes:
            self.engine.upload_pool(pack_pool(self._scenes))
        # spaces (envs/spaces.py:27-61 + wrappers)
        if env.action_mode == "discrete":
            self.single_action_space = Discrete(len(aspec["discrete_actions"]))
        else:
            self.single_action_space = Box(np.asarray(aspec["low"], np.float32), np.asarray(aspec["high"], np.float32),
                                           dtype=np.float32)
        F = env.frame_stack
        if obs_mode == E.OBS_SEMANTIC:
            C = E.MASK_CHANNELS[env.semantic_mask_ch]
            # FlattenStackedFrames | VehicleTemporalFusionWrapper | WeightedVehicleHistoryWrapper (envs/__init__.py:73-81)
            c_out = {"stack": F * C, "vehicle_temporal": C - 1 + 3, "vehicle_weighted": C}[self.fusion]
            if mask_dtype == "uint8" and self.fusion != "vehicle_weighted":
                self.single_observation_space = Box(0, 1, (c_out, *env.obs_size), np.uint8)
            else:
                self.single_observation_space = Box(0.0, 1.0, (c_out, *env.obs_size), np.float32)
        elif obs_mode == E.OBS_GRAY:
            self.single_observation_space = Box(0, 255, (F, *env.obs_size), np.uint8)
        else:
            self.single_observation_space = Box(0, 255, (env.size, env.size, 3), np.uint8)
        # wrap_env(eval=True) seeds the action space with 999, training envs with cfg.seed (envs/__init__.py:84-88)
        self.single_action_space.seed(999 if eval else cfg.seed)
        self.observation_space = self.single_observation_space  # batched spaces are not modelled; shapes are per env
        self.action_space = self.single_action_space
        self._act_pin = self._act_np = None  # pinned staging of host actions (allocated by the first step)
        self._needs_reset = np.ones(self.num_envs, dtype=bool)
        self._scene_of_env = np.zeros(self.num_envs, dtype=np.int64)
        self.current_hero = None
        self._generated, self._shipped_lists = {}, {}
        self._episode_t0 = np.full(self.num_envs, time.perf_counter())
        self.recorder, self._rec_pending_reset = None, False
        self._final_fused = None  # same_step with fusion: [N, *fused shape], rows of the envs that ended last step
        self._fused = []  # with fusion: two [N, *fused shape] buffers, filled in turn (`_fuse`)
        if getattr(cfg, "capture_video", False) and self.env_offset == 0:  # global env 0 only (envs/__init__.py:93-100)
            from .recorder import FrameRecorder

            self.recorder = FrameRecorder(cfg, eval=eval)
            self.engine.keep_fov(True)
            self.host_infos = True                   # the recorder needs env 0's done flag on the host

    @staticmethod
    def _crop_size(env) -> int:
        import math

        m = env.size - 1
        ax = max(0, min(m, int(round(m * env.ego_anchor_x_frac))))
        ay = max(0, min(m, int(round(m * env.ego_anchor_y_frac))))
        return max(env.size, int(math.ceil(2.0 * math.hypot(max(ax, m - ax), max(ay, m - ay)))))

    # ---------------------------------------------------------------- pool
    def _shipped_scenes(self, name):
        if name not in self._shipped_lists:
            self._shipped_lists[name] = load_shipped_pool(name)
        return self._shipped_lists[name]

    def _check_actor_capacity(self):
        need = max(len(s["act_kind"]) for s in self._scenes)
        if need > self.engine.cfg.max_actors:
            raise ValueError(f"scene with {need} actors exceeds the engine's max_actors={self.engine.cfg.max_actors} "
                             "(EnvConfig.max_vehicles + 2); raise max_vehicles")

    def set_scene_pool(self, scenes):
        """Replace the device-resident pool (list of scene dicts, see pool.py)."""
        self._scenes = list(scenes)
        self._pool_is_user = True
        self._generated = {}
        self.engine.invalidate()  # indices of the old pool mean nothing in the new one: every env resets first
        self._needs_reset[:] = True
        self.engine.upload_pool(pack_pool(self._scenes))

    def _scenes_from_options(self, options, mask):
        """Resolve reset options to pool indices, generating scripted scenes on the host if needed
        (the reference builds the scene inside reset: carlabev.py:96-148)."""
        n = self.num_envs
        if "scene_ids" in options:
            ids = np.broadcast_to(np.asarray(options["scene_ids"], dtype=np.int64), (n,)).copy()
            if ids.min() < 0 or ids.max() >= len(self._scenes):
                raise ValueError("scene_ids outside the scene pool")
            return ids
        scene = options.get("scene")
        authored = options.get("config_file") or (scene if str(scene).endswith(".json") else None)
        if authored is None and scene == "pool" and not self._scenes:
            raise RuntimeError("no scene pool: pass scenes=... / call set_scene_pool(), or reset with "
                               "options={'scene': 'rdm' | 'lead_brake' | 'jaywalk' | 'red_light_runner', ...}")
        if authored is None and (scene == "pool" or (scene is None and self._scenes and self._pool_is_user)):
            base = int(options.get("scene_seed", options.get("_vector_seed", self.env_cfg.seed)))
            return (base + self.env_offset + np.arange(n)) % len(self._scenes)
        if authored is None and scene is None:
            # the reference's default: SceneGenerator.build_scene(scene="rdm") seeded with cfg.seed
            # (scene_generator.py:97, carlabev.py:83-94)
            scene = "rdm"
            options = {**options, "scene": "rdm"}
        if authored is not None and not isinstance(authored, dict) and not os.path.exists(str(authored)):
            # the reference's own 7 scene files (assets/scenes/*.json) ship with the package, addressed by file name
            bundled = S.bundled_authored_files()
            if os.path.basename(str(authored)) not in bundled:
                raise FileNotFoundError(f"authored scene file {authored!r} not found (bundled: {sorted(bundled)})")
            options = {**options, "config_file": bundled[os.path.basename(str(authored))]}
        if authored is not None or scene in ("rdm", "lead_brake", "jaywalk", "red_light_runner"):
            # The reference builds the scene inside reset (carlabev.py:96-148); here the host generator
            # (scenes.py, bit-identical to the reference's post-reset state) fills the device pool on demand.
            # SyncVectorEnv passes the same options to every env: with options["scene_seed"] every env gets the
            # same scene; with reset(seed=s) env i is seeded s + i (gymnasium vector reset).
            if "scene_seed" in options:
                seeds = np.full(n, int(options["scene_seed"]), dtype=np.int64)
            elif "_vector_seed" in options:
                seeds = int(options["_vector_seed"]) + self.env_offset + np.arange(n, dtype=np.int64)
            else:
                seeds = np.full(n, int(self.env_cfg.seed), dtype=np.int64)
            base_opts = {k: v for k, v in options.items() if k not in ("scene_seed", "_vector_seed", "reset_mask")}
            key = repr(sorted((k, repr(v)) for k, v in base_opts.items()))
            cache = self._generated.setdefault(key, {})
            sel = np.ones(n, bool) if mask is None else np.asarray(mask, bool)
            new = [int(sd) for sd in np.unique(seeds[sel]) if int(sd) not in cache]
            if new:
                # snapshots exported from the reference with exactly these options (entry i <-> scene_seed i)
                shipped = None if authored is not None or self.env_cfg.size != 128 else \
                    shipped_pool_for(options, self.env_cfg.max_vehicles)  # exported at size 128 (spawn validation)
                ready = {}
                if shipped is not None:
                    pool = self._shipped_scenes(shipped)
                    ready = {sd: pool[sd] for sd in new if 0 <= sd < len(pool)}
                todo = [sd for sd in new if sd not in ready]
                built = S.build_pool([{**base_opts, "scene_seed": sd} for sd in todo], pad=self.pad,
                                     max_vehicles=self.env_cfg.max_vehicles, size=self.env_cfg.size)
                ready.update(zip(todo, built))
                for sd in new:
                    self._scenes.append(ready[sd])
                    cache[sd] = len(self._scenes) - 1
                self._check_actor_capacity()
                self.engine.upload_pool(pack_pool(self._scenes))
            ids = np.zeros(n, dtype=np.int64)
            ids[sel] = [cache[int(sd)] for sd in seeds[sel]]
            return ids
        raise KeyError(f"Unknown scenario '{scene}'")

    # ---------------------------------------------------------------- gym surface
    def reset(self, *, seed=None, options=None):
        t = self.torch
        options = {} if options is None else dict(options)
        mask = options.pop("reset_mask", None)
        if mask is not None:
            mask = np.asarray(mask)
            assert mask.dtype == np.bool_ and mask.shape == (self.num_envs,) and mask.any(), \
                "reset_mask must be a bool array of shape (num_envs,) with at least one True"
        if seed is not None and "scene_seed" not in options:
            # gymnasium SyncVectorEnv.reset(seed=s) seeds env i with s + i; CarlaBEV._resolve_rng_bundle then uses it
            # as the scene seed (carlabev.py:83-94)
            options["_vector_seed"] = int(seed)
        ids = self._scenes_from_options(options, mask)
        first = bool(self._needs_reset.all()) and self.engine.head < 0
        if first and mask is not None and not mask.all():
            raise RuntimeError("the first reset must cover every env")
        m = None if (mask is None or mask.all()) else mask
        obs = self.engine.reset(ids, m)
        if self.fusion != "stack":
            obs = self._fuse()
        if m is None:
            self._needs_reset[:] = False
            self._scene_of_env[:] = ids
            self._episode_t0[:] = time.perf_counter()
        else:
            self._needs_reset[m] = False
            self._scene_of_env[m] = ids[m]
            self._episode_t0[m] = time.perf_counter()
        if self.recorder is not None and (m is None or m[0]):
            self.recorder.on_reset(self.engine.fov()[0].cpu().numpy())
        infos = self._reset_infos(np.ones(self.num_envs, bool) if m is None else m) if self.host_infos else {}
        return self._out_obs(obs), infos

    def _reset_infos(self, mask):
        """CarlaBEV.reset's info (carlabev.py:145-148) batched the way gymnasium's vector envs do (`key` array +
        `_key` mask, nested dicts recursively): the scenario context that is a property of the scene (kind, level,
        seed, route length, traffic count) and the spawn validation, which every pool entry has passed."""
        from .pool import SCENE_KINDS

        n = self.num_envs
        idx = np.flatnonzero(mask)
        sc = [self._scenes[int(self._scene_of_env[i])] for i in idx]

        def col(values, dtype):
            a = np.full(n, None, dtype=object) if dtype is object else np.zeros(n, dtype=dtype)
            a[idx] = values
            return a

        scenario = {
            "scene": col([SCENE_KINDS[int(s["kind"])] if 0 <= int(s["kind"]) < len(SCENE_KINDS) else "rdm" for s in sc], object),
            "level": col([int(s["level"]) for s in sc], np.int64),
            "scene_seed": col([int(s["seed"]) for s in sc], np.int64),
            "route_length_m": col([float(s["len_ego_route"]) for s in sc], np.float64),
            "scenario_param_num_vehicles": col([int(s["num_vehicles"]) for s in sc], np.int64),
        }
        scenario.update({f"_{k}": mask.copy() for k in list(scenario)})
        spawn = {"valid": col([True] * len(idx), np.bool_), "reason": col(["ok"] * len(idx), object)}
        spawn.update({f"_{k}": mask.copy() for k in list(spawn)})
        return {"scenario": scenario, "_scenario": mask.copy(), "spawn_validation": spawn, "_spawn_validation": mask.copy()}

    def step(self, actions):
        """SyncVectorEnv.step (envs/__init__.py:116-119 -> carlabev.py:223-231) for every env of the shard.

        `actions` may be a host array (NumPy / list, like the reference's callers pass) or a CUDA tensor.  With host
        infos on, rewards / flags / terminal summaries come to the host through one pinned D2H copy that overlaps the
        raster kernel, and `step` returns as soon as THEY have landed: the observation is a device tensor whose
        producer may still be running on the current stream (anything enqueued on that stream afterwards is ordered).
        The stacked observation is a zero-copy view of the frame ring: it stays valid for `engine.L - 2 * frame_stack
        + 1` further calls (>= 1 with the default ring of >= 2 * frame_stack slots), then the head or its mirror
        write reaches its oldest slot.  A reset of an env -- the auto-reset of "next_step" or "same_step", a masked
        `reset`, a `restore` -- rewrites that env's window slots at that call's head, so every view of the env that
        shares them changes.  Under "same_step" that is the previous call's `obs` of every env that ends in this
        call: store `obs` (copy it into the rollout buffer) before calling `step`, or clone it.  A fused observation
        (`temporal_fusion_mode`) is a copy, not a view: two buffers are filled in turn, so the previous call's `obs`
        stays intact through this call and is overwritten by the next.  Clone what must live longer."""
        t = self.torch
        if self.autoreset == "disabled" and self._needs_reset.any():
            # gymnasium SyncVectorEnv(AutoresetMode.DISABLED) asserts on this
            raise AssertionError(f"step() on terminated envs {np.flatnonzero(self._needs_reset).tolist()}; "
                                 "call reset(options={'reset_mask': ...}) first")
        eng = self.engine
        discrete = self.env_cfg.action_mode == "discrete"
        on_device = isinstance(actions, t.Tensor) and actions.is_cuda
        if on_device:
            a = actions.to(t.int64).contiguous().view(self.num_envs) if discrete else \
                actions.to(t.float32).contiguous().view(self.num_envs, 3)
            if self.host_infos:
                eng.step_host_full(a)
            else:
                eng.step(a)
        elif not self.host_infos:
            # fully asynchronous mode: the host never waits for the device, so a pinned staging buffer could be
            # overwritten while an earlier step's copy is still queued -- take a stream-ordered copy of the actions
            a = t.as_tensor(np.asarray(actions), dtype=t.int64 if discrete else t.float32).to(self.device)
            eng.step(a.view(self.num_envs) if discrete else a.view(self.num_envs, 3))
        else:
            if self._act_pin is None:
                self._act_pin = (t.zeros(self.num_envs, dtype=t.int64) if discrete
                                 else t.zeros(self.num_envs, 3, dtype=t.float32)).pin_memory()
                self._act_np = self._act_pin.numpy()
            # safe to overwrite: the previous step waited for its host outputs, which follow its H2D copy
            self._act_np[...] = np.asarray(actions).reshape(self._act_np.shape)
            eng.step_host_full(self._act_pin, episode=True)
        obs = eng.obs() if self.fusion == "stack" else self._fuse()
        rew, term, trunc = eng.reward, eng.terminated.view(t.bool), eng.truncated.view(t.bool)
        self.current_hero = eng.hero
        infos = {"hero": eng.hero, "cause": eng.cause}
        if not self.host_infos:
            # fully asynchronous step: terminal summaries stay on the device (rows of finished envs are valid)
            infos["episode_block"] = eng.episode
            if self.autoreset == "same_step":  # dense: rows of the envs that ended are valid
                infos["final_obs"], infos["_final_obs"] = eng.final_obs, term | trunc
            return obs, rew, term, trunc, infos
        eng.wait_host_outputs()  # reward / flags / episode block are on the host; the raster kernel may still run
        term_h = eng.host_terminated.numpy().view(np.bool_)
        trunc_h = eng.host_truncated.numpy().view(np.bool_)
        done_host = term_h | trunc_h
        if self.recorder is not None:
            self._record_step(bool(done_host[0]))
        if done_host.any():
            if self.autoreset == "same_step":
                # gymnasium SAME_STEP: the terminal keys move under final_info, next to the terminal observation
                infos.update(self._final_obs_infos(done_host))
                infos["final_info"], infos["_final_info"] = self._terminal_infos(done_host), done_host.copy()
            else:
                infos.update(self._terminal_infos(done_host))
            if self.autoreset == "disabled":
                self._needs_reset |= done_host
        if self.to_numpy:
            return (self._out_obs(obs), eng.host_reward.numpy().copy(), term_h.copy(), trunc_h.copy(), infos)
        return obs, rew, term, trunc, infos

    def _terminal_infos(self, done_host):
        """episode_info (stats.py:127-148 + carlabev.py:177-185) and RecordEpisodeStatistics' `episode`
        (r = sum of rewards, l = steps: the same numbers as the summary's return / length).  With an action repeat K,
        `length` counts simulator steps and `l` agent steps: ceil(length / K), since every agent step of an episode but
        its last takes K simulator steps.  Built from the pinned host copy of the episode block with a handful of
        vectorised NumPy operations."""
        idx = np.flatnonzero(done_host)
        ep = self.engine.host_episode.numpy()[idx]
        n = self.num_envs
        mask = done_host.copy()
        cols = np.zeros((len(E.EPISODE_FIELDS), n), dtype=np.float64)
        cols[:, idx] = ep.T
        episode_info = {}
        for k, name in enumerate(E.EPISODE_FIELDS):
            if name == "cause":
                col = np.full(n, None, dtype=object)
                col[idx] = _CAUSE_ARRAY[ep[:, k].astype(np.int64)]
                name = "termination"
            elif name == "length":
                col = cols[k].astype(np.int64)
            else:
                col = cols[k]
            episode_info[name] = col
            episode_info[f"_{name}"] = mask
        now = time.perf_counter()  # RecordEpisodeStatistics' `t`: wall-clock seconds since the episode began
        tm = np.zeros(n)
        tm[idx] = np.round(now - self._episode_t0[idx], 6)
        self._episode_t0[idx] = now   # device auto-reset: the next episode of these envs starts now
        K = self.action_repeat
        length = episode_info["length"]
        return {"episode_info": episode_info, "_episode_info": mask,
                "episode": {"r": episode_info["return"], "_r": mask, "l": length if K == 1 else (length + K - 1) // K,
                            "_l": mask,
                            "t": tm, "_t": mask}, "_episode": mask}

    def _final_obs_infos(self, done_host):
        """`final_obs` / `_final_obs` of autoreset="same_step": the windows the finished envs' episodes ended on.  On the
        device the dense [N, ...] buffer (rows of finished envs valid), fused with temporal_fusion_mode from the k
        finished windows only; with to_numpy an object array, each finished env's array and None elsewhere."""
        t, eng = self.torch, self.engine
        idx = np.flatnonzero(done_host)
        final = eng.final_obs
        sel = None
        if self.fusion != "stack" or self.to_numpy:
            sel = t.from_numpy(idx).to(self.device)
        if self.fusion != "stack":
            if self._final_fused is None:
                code = E.FUSE_MODES[self.fusion]
                self._final_fused = t.zeros(self.num_envs, *eng._fused_shape(code), dtype=eng._fused_dtype(code),
                                            device=self.device)
            fused = eng.fuse_windows(self.fusion, final.index_select(0, sel))
            final = self._final_fused.index_copy_(0, sel, fused)
        if self.to_numpy:
            rows = final.index_select(0, sel).cpu().numpy()
            out = np.full(self.num_envs, None, dtype=object)
            for k, i in enumerate(idx):
                out[i] = rows[k]
            final = out
        return {"final_obs": final, "_final_obs": done_host.copy()}

    def _record_step(self, done0):
        rec = self.recorder
        if self.autoreset == "next_step" and self._rec_pending_reset:
            # this step consumed env 0's device auto-reset: its frame is the reset frame of a new episode
            rec.on_reset(self.engine.fov()[0].cpu().numpy())
        elif rec.frames is not None:
            rec.on_step(self.engine.fov()[0].cpu().numpy(), done0)
        self._rec_pending_reset = done0 and self.autoreset == "next_step"

    def _fuse(self):
        """The fused observation, written into the older of two buffers: the one returned by the previous call stays
        intact through this one (`obs` and `next_obs` of a transition are both valid)."""
        if not self._fused:
            code = E.FUSE_MODES[self.fusion]
            shape, dtype = (self.num_envs, *self.engine._fused_shape(code)), self.engine._fused_dtype(code)
            self._fused = [self.torch.empty(shape, dtype=dtype, device=self.device) for _ in range(2)]
        self._fused.reverse()
        return self.engine.fuse(self.fusion, out=self._fused[0])

    def _out_obs(self, obs):
        return obs.cpu().numpy() if self.to_numpy else obs

    # ---------------------------------------------------------------- snapshot / restore
    def snapshot(self, env_ids=None):
        """Device-side snapshot of envs `env_ids` of this shard (default: all; indices are local to the shard), see
        `Engine.snapshot`.  The wall-clock start of each env's episode is kept with it for RecordEpisodeStatistics' `t`."""
        snap = self.engine.snapshot(env_ids)
        snap.episode_t0 = self._episode_t0[self._host_index(env_ids, snap.n_rows)].copy()
        return snap

    def restore(self, snap, env_ids=None, rows=None):
        """Write snapshot rows into envs (see `Engine.restore`) and return their observation -- fused when
        `temporal_fusion_mode` asks for it.  The host bookkeeping follows the restored rows (terminal envs need a reset
        under autoreset "disabled", reset infos name the restored scene); that costs one small device-to-host copy.
        The window frames are rewritten in place, so an observation view still held for these envs changes."""
        if self.recorder is not None:
            raise ValueError("restore() is not available while capture_video records env 0's episodes")
        obs = self.engine.restore(snap, env_ids, rows)
        n = len(rows) if rows is not None else (len(env_ids) if env_ids is not None else snap.n_rows)
        ids_h = self._host_index(env_ids, n)
        rows_h = self._host_index(rows, n)
        hdr = snap.header().cpu().numpy()[rows_h]  # scene, episode, done of the restored rows
        if self.autoreset == "disabled":
            self._needs_reset[ids_h] = hdr[:, 2] != 0
        self._scene_of_env[ids_h] = hdr[:, 0]
        t0 = getattr(snap, "episode_t0", None)
        self._episode_t0[ids_h] = t0[rows_h] if t0 is not None else time.perf_counter()
        if self.fusion != "stack":
            obs = self._fuse()
        return self._out_obs(obs)

    def _host_index(self, idx, n):
        if idx is None:
            return np.arange(n)
        if isinstance(idx, self.torch.Tensor):
            idx = idx.cpu()
        return np.asarray(idx, dtype=np.int64)

    def vector_observation(self):
        """The reference's `obs_mode="vector"` observation of every env (envs/carlabev.py:237-244):
        float32 [N, 7] = hero.state (x, y, yaw, v) ++ set_point (x, y, yaw).  Valid after a step."""
        h = self.engine.hero
        return self.torch.cat([h[:, 0:4], h[:, 9:12]], dim=1).to(self.torch.float32)

    def episode_statistics(self, reset=False):
        """Device-accumulated episode statistics (CBEV_S_* of include/cbev.h) as a CUDA float64 tensor.
        This vector is the only thing ranks exchange (carlabev_env_b200.distributed.allreduce_stats)."""
        return self.engine.read_stats(reset)

    def close(self):
        if self.recorder is not None:
            self.recorder.flush()
        self.engine.close()


def make_env(cfg=None, eval: bool = False, **engine_kwargs) -> CarlaBEVVectorEnv:  # noqa: A002
    """envs/__init__.py:108-120.  Multi-GPU: one process per GPU, `make_env(cfg, shard=(rank, world_size),
    device=local_rank)` gives each its contiguous slice of the `cfg.num_envs` environments; no collective is
    involved in stepping (`distributed.allreduce_stats` sums the episode statistics when asked)."""
    if cfg is None:
        cfg = RunConfig()
    if not hasattr(cfg, "env") and not (isinstance(cfg, dict) and "env" in cfg):
        cfg = validate_run_config({"env": cfg})
    else:
        cfg = validate_run_config(cfg)
    return CarlaBEVVectorEnv(cfg, eval=eval, **engine_kwargs)

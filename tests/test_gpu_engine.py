"""GPU tests of the engine beyond golden replay: batched parity with the oracle on fresh scenes, the
observation ring (wrap + mirror), masked reset, device auto-reset, the VectorEnv surface, error paths and
size-independent properties at the benchmark size (4096 envs)."""
import os

import numpy as np
import pytest

from golden_util import load_map

pytestmark = pytest.mark.gpu


def _scenes(kinds, seed0=500):
    from carlabev_env_b200.scenes import build_scripted_scene

    cls = load_map()
    return [build_scripted_scene(k, seed0 + i, level=lv, cls_map=cls) for i, (k, lv) in enumerate(kinds)]


def _engine(n, scenes, **kw):
    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.pool import pack_pool

    args = dict(obs_mode=E.OBS_SEMANTIC, mask_mode="6-class", frame_stack=4, action_mode=E.ACTION_CONTINUOUS,
                max_actors=4, ring_budget_bytes=64 << 20)
    args.update(kw)
    eng = E.Engine(n, **args)
    eng.upload_map(load_map())
    eng.upload_pool(pack_pool(scenes))
    return eng


def _rand_actions(rng, n):
    return np.stack([rng.uniform(0, 1, n), rng.uniform(-1, 1, n), rng.uniform(0, 1, n)], axis=1).astype(np.float32)


def _check_env(t, i, hero, rew, term, obs, oracle, out):
    o, r, te, tr, _ = out
    e = oracle.sim.ego
    assert np.allclose(hero[:4], [e.x, e.y, e.yaw, e.v], rtol=1e-9, atol=1e-9), (t, i, "pose")
    assert abs(r - rew) < 1e-9, (t, i, "reward", r, rew)
    assert te == term, (t, i, "terminated")
    assert np.array_equal(obs, o), (t, i, "observation")


def test_batched_parity_with_masked_resets():
    import torch

    from oracle.env import OracleEnv

    kinds = [("lead_brake", 1 + i % 3) for i in range(10)] + [("jaywalk", 1 + i % 4) for i in range(10)]
    scenes = _scenes(kinds)
    n = len(scenes)
    eng = _engine(n, scenes)
    oracles = [OracleEnv(load_map(), action_mode="continuous") for _ in range(n)]
    scene_of = np.arange(n)
    obs = eng.reset(torch.arange(n, dtype=torch.int32)).cpu().numpy()
    for i in range(n):
        assert np.array_equal(obs[i], oracles[i].reset(scenes[i]))
    rng = np.random.default_rng(1)
    n_resets = 0
    for t in range(60):
        a = _rand_actions(rng, n)
        if t < 25:
            a[n // 2:, 0] *= 0.2  # let the pedestrians' FSM play out for part of the batch
        eng.step(torch.from_numpy(a).cuda())
        obs, rew = eng.obs().cpu().numpy(), eng.reward.cpu().numpy()
        term, hero = eng.terminated.cpu().numpy().astype(bool), eng.hero.cpu().numpy()
        for i in range(n):
            _check_env(t, i, hero[i], rew[i], term[i], obs[i], oracles[i], oracles[i].step(a[i]))
        if term.any():  # SyncVectorEnv-style masked reset with a new scene for the finished envs
            scene_of[term] = (scene_of[term] + 7) % n
            obs = eng.reset(torch.from_numpy(scene_of.astype(np.int32)), term).cpu().numpy()
            for i in np.flatnonzero(term):
                assert np.array_equal(obs[i], oracles[i].reset(scenes[scene_of[i]])), (t, i, "masked reset obs")
                n_resets += 1
            for i in np.flatnonzero(~term):  # untouched envs keep their window
                assert np.array_equal(obs[i], oracles[i]._stacked()), (t, i, "window of a non-reset env")
    assert n_resets > 0
    eng.close()


@pytest.mark.parametrize("ring_slots", [7, 9])
def test_ring_wrap_keeps_the_frame_stack(ring_slots):
    import torch

    from oracle.env import OracleEnv

    scenes = _scenes([("jaywalk", 2), ("jaywalk", 1), ("lead_brake", 2)], seed0=900)
    eng = _engine(3, scenes, ring_slots=ring_slots)
    oracles = [OracleEnv(load_map(), action_mode="continuous") for _ in range(3)]
    eng.reset(torch.arange(3, dtype=torch.int32))
    for i in range(3):
        oracles[i].reset(scenes[i])
    alive = np.ones(3, bool)
    for t in range(3 * ring_slots + 2):
        a = np.tile(np.array([[0.0, 0.0, 1.0]], np.float32), (3, 1))  # brake: long episodes
        eng.step(torch.from_numpy(a).cuda())
        obs = eng.obs().cpu().numpy()
        for i in range(3):
            if alive[i]:
                o, _, te, _, _ = oracles[i].step(a[i])
                assert np.array_equal(obs[i], o), (t, i, eng.head)
                alive[i] = not te
    assert alive.any()
    eng.close()


def _splitmix64(z):
    m = (1 << 64) - 1
    z = (z + 0x9E3779B97F4A7C15) & m
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & m
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & m
    return z ^ (z >> 31)


def test_device_autoreset_next_step():
    import torch

    from carlabev_env_b200 import engine as E
    from oracle.env import OracleEnv

    kinds = [("lead_brake", 1 + i % 3) for i in range(12)]
    scenes = _scenes(kinds, seed0=300)
    n, seed = 12, 5
    eng = _engine(n, scenes, autoreset=E.AUTORESET_NEXT_STEP, seed=seed)
    oracles = [OracleEnv(load_map(), action_mode="continuous") for _ in range(n)]
    eng.reset(torch.arange(n, dtype=torch.int32))
    for i in range(n):
        oracles[i].reset(scenes[i])
    done = np.zeros(n, bool)
    episodes = np.zeros(n, dtype=np.int64)
    rng = np.random.default_rng(2)
    n_auto = 0
    m = (1 << 64) - 1
    for t in range(70):
        a = _rand_actions(rng, n)
        a[:, 0] = np.clip(a[:, 0] + 0.3, 0, 1)
        eng.step(torch.from_numpy(a).cuda())
        obs, rew = eng.obs().cpu().numpy(), eng.reward.cpu().numpy()
        term, hero = eng.terminated.cpu().numpy().astype(bool), eng.hero.cpu().numpy()
        for i in range(n):
            if done[i]:  # gymnasium NEXT_STEP: this step resets, ignores the action, reward 0, not terminated
                h = _splitmix64((seed + i * 0x9E3779B97F4A7C15 + int(episodes[i]) * 0xD1B54A32D192ED03) & m)
                sc = h % len(scenes)
                assert int(hero[i][E.HERO_FIELDS.index("scene")]) == sc, (t, i)
                assert rew[i] == 0.0 and not term[i]
                assert np.array_equal(obs[i], oracles[i].reset(scenes[sc])), (t, i, "auto-reset obs")
                done[i] = False
                n_auto += 1
            else:
                _check_env(t, i, hero[i], rew[i], term[i], obs[i], oracles[i], oracles[i].step(a[i]))
                if term[i]:
                    done[i] = True
                    episodes[i] += 1
    assert n_auto > 3
    stats = eng.read_stats().cpu().numpy()
    assert stats[0] == episodes.sum() and stats[-1] == 70 * n
    eng.close()


def test_vector_env_surface_and_infos():
    import torch

    from carlabev_env_b200 import EnvConfig, RunConfig, make_env

    scenes = _scenes([("lead_brake", 1 + i % 3) for i in range(6)], seed0=40)
    cfg = RunConfig(env=EnvConfig(action_mode="continuous"), num_envs=6)
    envs = make_env(cfg, scenes=scenes, ring_budget_bytes=64 << 20)
    assert envs.num_envs == 6 and envs.single_observation_space.shape == (24, 96, 96)
    assert envs.single_action_space.shape == (3,)
    obs, infos = envs.reset(options={"scene_ids": np.arange(6)})
    assert obs.shape == (6, 24, 96, 96) and obs.dtype == torch.float32
    assert infos["scenario"]["scene"].tolist() == ["lead_brake"] * 6 and infos["_spawn_validation"].all()
    with pytest.raises(AssertionError):
        envs.reset(options={"reset_mask": np.zeros(6, bool)})
    finished = None
    for t in range(80):
        a = np.tile(np.array([[1.0, 0.3, 0.0]], np.float32), (6, 1))
        obs, rew, term, trunc, infos = envs.step(a)
        assert rew.dtype == torch.float64 and term.dtype == torch.bool and infos["hero"].shape == (6, 32)
        if bool((term | trunc).any()):
            finished = (term | trunc).cpu().numpy()
            ei = infos["episode_info"]
            assert np.array_equal(infos["_episode_info"], finished)
            i = int(np.flatnonzero(finished)[0])
            assert ei["termination"][i] in ("collision", "success", "out_of_bounds")
            assert ei["length"][i] == infos["episode"]["l"][i] == t + 1
            assert abs(ei["return"][i] - infos["episode"]["r"][i]) < 1e-9
            break
    assert finished is not None
    vec = envs.vector_observation()  # obs_mode="vector" of the base env: state ++ set_point, float32 (7,)
    assert vec.shape == (6, 7) and vec.dtype == torch.float32
    assert torch.equal(vec[:, :4], infos["hero"][:, :4].float())
    with pytest.raises(AssertionError):  # SyncVectorEnv(AutoresetMode.DISABLED) refuses to step finished envs
        envs.step(np.zeros((6, 3), np.float32))
    obs, _ = envs.reset(options={"scene_ids": np.arange(6), "reset_mask": finished})
    envs.step(np.zeros((6, 3), np.float32))
    # scripted scene built on the host at reset time, like the reference's reset(options={"scene": ...})
    obs, rinfo = envs.reset(options={"scene": "jaywalk", "level": 3, "scene_seed": 11})
    assert obs.shape == (6, 24, 96, 96)
    assert rinfo["scenario"]["scene"].tolist() == ["jaywalk"] * 6 and rinfo["scenario"]["level"].tolist() == [3] * 6
    assert rinfo["scenario"]["scene_seed"].tolist() == [11] * 6 and rinfo["_scenario"].all()
    assert rinfo["spawn_validation"]["valid"].all() and rinfo["spawn_validation"]["reason"][0] == "ok"
    assert len(set(envs._scene_of_env.tolist())) == 1            # options["scene_seed"]: the same scene for every env
    obs, _ = envs.reset(seed=40, options={"scene": "lead_brake", "level": 1})
    assert len(set(envs._scene_of_env.tolist())) == 6            # reset(seed=s): env i is seeded s + i
    from carlabev_env_b200 import reset as R

    obs, _ = envs.reset(seed=3, options=R.build_reset_options(R.RandomNavigationReset(difficulty_id="rt_medium_v1")))
    assert len(set(envs._scene_of_env.tolist())) == 6
    # seeds outside the shipped snapshots are generated on the host (lane graphs + shortest paths, scenes.py)
    obs, _ = envs.reset(seed=1000, options={"scene": "rdm", "num_vehicles": 3, "route_dist_range": [30, 60]})
    assert len(set(envs._scene_of_env.tolist())) == 6
    assert max(len(envs._scenes[i]["act_kind"]) for i in envs._scene_of_env) <= 3
    obs, _ = envs.reset(options={"scene": "red_light_runner", "scene_seed": 77})
    envs.step(np.zeros((6, 3), np.float32))
    with pytest.raises(RuntimeError):
        envs.reset(options={"scene": "rdm", "route_profile": "left_turn", "max_route_attempts": 1, "scene_seed": 1})
    obs, _ = envs.reset(seed=20, options={"scene": "rdm", "num_vehicles": 2, "route_profile": "single_left",
                                          "route_dist_range": [30, 130]})
    # authored scene file (bundled, addressed by name) and a typed preset request (config/reset.py mirror)
    obs, _ = envs.reset(options=R.build_reset_options(R.AuthoredSceneReset("redlightrunner-01.01.json", True, 2)))
    assert len(envs._scenes[envs._scene_of_env[0]]["tl_color"]) >= 2
    envs.step(np.zeros((6, 3), np.float32))
    obs, _ = envs.reset(seed=5, options=R.build_reset_options(R.ScenarioPresetReset("lead_brake_debug")))
    assert len(set(envs._scene_of_env.tolist())) == 6
    with pytest.raises(FileNotFoundError):
        envs.reset(options={"config_file": "no_such_scene.json"})
    envs.close()


def test_error_paths():
    import torch

    from carlabev_env_b200 import engine as E

    scenes = _scenes([("lead_brake", 1)])
    with pytest.raises(E.CbevError, match="ring_slots"):
        _engine(2, scenes, ring_slots=4)
    eng = _engine(2, scenes)
    with pytest.raises(E.CbevError, match="before reset"):
        eng.step(torch.zeros(2, 3, device="cuda"))
    with pytest.raises(E.CbevError, match="first reset"):
        eng.reset(torch.zeros(2, dtype=torch.int32), np.array([True, False]))
    big = _scenes([("lead_brake", 3)])
    small = E.Engine(1, action_mode=E.ACTION_CONTINUOUS, max_actors=1, ring_budget_bytes=32 << 20)
    from carlabev_env_b200.pool import pack_pool

    with pytest.raises(E.CbevError, match="max_actors"):
        small.upload_pool(pack_pool(big))
    eng.close()
    small.close()


def test_debug_flags_reject_unknown_bits():
    from carlabev_env_b200 import engine as E

    eng = _engine(2, _scenes([("lead_brake", 1)]))
    for bad in (8, 16, 64, 1 << 20):  # 8 / 16 / 64 selected store variants of k_render that no longer exist
        with pytest.raises(E.CbevError, match="accepted bits: 1, 2, 4, 32, 128, 256, 512"):
            eng.set_debug_flags(bad)
    for bit in (1, 2, 4, 32, 128, 256, 512):
        eng.set_debug_flags(bit)
    eng.set_debug_flags(0)
    eng.close()


def test_full_size_properties():
    """BASELINE configs[1] size (4096 envs): determinism, mask structure and the frame-stack shift property."""
    import torch

    from carlabev_env_b200 import engine as E

    scenes = _scenes([("lead_brake", 1 + i % 3) for i in range(64)], seed0=2000)
    n = 4096

    def run():
        eng = _engine(n, scenes, autoreset=E.AUTORESET_NEXT_STEP, seed=9, ring_budget_bytes=12 << 30)
        eng.reset(torch.arange(n, dtype=torch.int32) % len(scenes))
        g = torch.Generator(device="cpu").manual_seed(0)
        prev, sums = None, []
        for t in range(12):
            a = torch.rand(n, 3, generator=g)
            a[:, 1] = a[:, 1] * 2 - 1
            eng.step(a.cuda())
            obs = eng.obs()
            assert obs.shape == (n, 24, 96, 96)
            assert bool(((obs == 0) | (obs == 1)).all())
            new = obs[:, 18:]
            excl = new[:, 0] + new[:, 1] + new[:, 2] + new[:, 3] + new[:, 4]  # one base class per pixel at most
            assert float(excl.max()) <= 1.0
            assert bool((new[:, 5] <= new[:, 1]).all())                       # route pixels count as drivable
            if prev is not None:
                keep = ~was_done                                               # noqa: F821
                assert bool((obs[keep, :18] == prev[keep, 6:]).all())          # stack shifts by one frame
            prev = obs.clone()
            was_done = eng.terminated.bool().clone()                           # these envs auto-reset next step
            sums.append(float(obs.sum()) + float(eng.reward.sum()))
        eng.close()
        return sums

    assert run() == run()


def test_rdm_and_red_light_pools_discrete_parity():
    """Scenes exported from the reference's graph-based generators (shipped pools): 25-vehicle random traffic and
    red_light_runner (traffic-light strips), discrete9 actions, 7-class masks."""
    import torch

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.config import ACTION_PROFILES
    from carlabev_env_b200.pool import load_shipped_pool, pack_pool
    from oracle.env import OracleEnv

    scenes = load_shipped_pool("rdm_rt_hard_v1")[:10] + load_shipped_pool("red_light_runner")[:2]
    n = len(scenes)
    eng = E.Engine(n, obs_mode=E.OBS_SEMANTIC, mask_mode="7-class", frame_stack=4, action_mode=E.ACTION_DISCRETE,
                   discrete_table=ACTION_PROFILES["discrete9_v1"]["discrete_actions"], max_actors=25,
                   ring_budget_bytes=64 << 20)
    eng.upload_map(load_map())
    eng.upload_pool(pack_pool(scenes))
    oracles = [OracleEnv(load_map(), semantic_mask_ch="7-class") for _ in range(n)]
    obs = eng.reset(torch.arange(n, dtype=torch.int32)).cpu().numpy()
    for i in range(n):
        assert np.array_equal(obs[i], oracles[i].reset(scenes[i]))
    rng = np.random.default_rng(4)
    alive = np.ones(n, bool)
    for t in range(90):
        a = rng.choice([1, 1, 1, 3, 4, 0, 5, 6], size=n)  # mostly throttle, some steering
        eng.step(torch.from_numpy(a).cuda())
        obs, rew = eng.obs().cpu().numpy(), eng.reward.cpu().numpy()
        term, hero = eng.terminated.cpu().numpy().astype(bool), eng.hero.cpu().numpy()
        ego, act = eng.get_state(25)
        for i in range(n):
            if not alive[i]:
                continue
            _check_env(t, i, hero[i], rew[i], term[i], obs[i], oracles[i], oracles[i].step(a[i]))
            ref = np.array([[b.x, b.y, b.yaw, b.v] for b in oracles[i].sim.actors])
            assert np.allclose(act[i, :len(ref), :4], ref, rtol=1e-9, atol=1e-9), (t, i, "actors")
            alive[i] = not term[i]
        if not alive.any():
            break
    assert t > 20
    eng.close()


@pytest.mark.parametrize("variant", ["plain", "fov_masked", "generic_rotate", "keep_frame"])
def test_raw_rgb_lookahead_dense_traffic(variant):
    """BASELINE configs[4] shape: raw (128, 128, 3) uint8 frames, lookahead_75 camera, 50 vehicles, continuous.  Variants:
    the corner mask, the range-tested rotate (debug flag 1) and the debug copy of the palette frame on the RGB path."""
    import torch

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.pool import load_shipped_pool, pack_pool
    from oracle.env import OracleEnv

    scenes = load_shipped_pool("rdm_dense_50")[:8]
    n = len(scenes)
    eng = E.Engine(n, obs_mode=E.OBS_RGB, action_mode=E.ACTION_CONTINUOUS, max_actors=50, anchor=(0.5, 0.75))
    eng.upload_map(load_map())
    eng.upload_pool(pack_pool(scenes))
    masked = variant == "fov_masked"
    if masked:
        from carlabev_env_b200.fovmask import corner_mask

        eng.upload_fov_mask(corner_mask(128, 0.5))
    if variant == "generic_rotate":
        eng.set_debug_flags(1)
    if variant == "keep_frame":
        eng.keep_fov(True)
    oracles = [OracleEnv(load_map(), obs_mode="bev_raw", frame_stack=1, action_mode="continuous", anchor=(0.5, 0.75),
                         fov_masked=masked) for _ in range(n)]
    obs = eng.reset(torch.arange(n, dtype=torch.int32)).cpu().numpy()
    assert obs.shape == (n, 128, 128, 3) and obs.dtype == np.uint8
    for i in range(n):
        assert np.array_equal(obs[i], oracles[i].reset(scenes[i])[0])
    rng = np.random.default_rng(6)
    alive = np.ones(n, bool)
    for t in range(50):
        a = _rand_actions(rng, n)
        a[:, 0] = np.clip(a[:, 0] + 0.3, 0, 1)
        a[:, 2] *= 0.2
        eng.step(torch.from_numpy(a).cuda())
        obs, rew = eng.obs().cpu().numpy(), eng.reward.cpu().numpy()
        term, hero = eng.terminated.cpu().numpy().astype(bool), eng.hero.cpu().numpy()
        for i in range(n):
            if not alive[i]:
                continue
            o, r, te, tr, _ = oracles[i].step(a[i])
            e = oracles[i].sim.ego
            assert np.allclose(hero[i][:4], [e.x, e.y, e.yaw, e.v], rtol=1e-9, atol=1e-9), (t, i)
            assert abs(r - rew[i]) < 1e-9 and te == term[i], (t, i)
            assert np.array_equal(obs[i], o[0]), (t, i, "rgb frame")   # bar: within 1 LSB; we get exact
            alive[i] = not te
        if variant == "keep_frame":
            from oracle import raster

            fr = eng.fov().cpu().numpy()
            assert all(np.array_equal(raster.PALETTE[fr[i]], obs[i]) for i in range(n)), (t, "palette frame")
    eng.close()


def test_pose_drift_over_1000_steps():
    """BASELINE north_star: poses within 1e-5 relative after 1000 steps on identical seeds and actions.
    A route-following policy (Stanley steering + speed hold, computed on the oracle state) keeps three
    16-vehicle random-traffic episodes alive for up to 1000 steps; the engine is free-running."""
    import torch

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.pool import load_shipped_pool, pack_pool
    from oracle.env import OracleEnv

    pool = load_shipped_pool("rdm_rt_medium_v1")
    scenes = [pool[16], pool[19], pool[8]]
    n = len(scenes)
    eng = E.Engine(n, obs_mode=E.OBS_SEMANTIC, mask_mode="6-class", frame_stack=4, action_mode=E.ACTION_CONTINUOUS,
                   max_actors=16, ring_budget_bytes=64 << 20)
    eng.upload_map(load_map())
    eng.upload_pool(pack_pool(scenes))
    eng.keep_fov(True)
    eng.reset(torch.arange(n, dtype=torch.int32))
    oracles = [OracleEnv(load_map(), action_mode="continuous", obs_mode="bev_raw", frame_stack=1) for _ in range(n)]
    for o, s in zip(oracles, scenes):
        o.reset(s)

    def policy(env, vt=2.8):
        e = env.sim.ego
        delta, _ = e.stanley()
        steer_deg = float(np.clip(18.0 / (1.0 + 0.35 * abs(e.v)), 8.0, 18.0))
        return np.array([np.clip(0.6 * (vt - e.v), 0, 1), np.clip(float(delta) / np.radians(steer_deg), -1, 1),
                         np.clip(0.3 * (e.v - vt - 0.5), 0, 1)], dtype=np.float32)

    alive = np.ones(n, bool)
    worst = 0.0
    steps_alive = np.zeros(n, int)
    for t in range(1000):
        a = np.stack([policy(o) if alive[i] else np.zeros(3, np.float32) for i, o in enumerate(oracles)])
        eng.step(torch.from_numpy(a).cuda())
        hero = eng.hero.cpu().numpy()
        term = eng.terminated.cpu().numpy().astype(bool)
        rew = eng.reward.cpu().numpy()
        for i in range(n):
            if not alive[i]:
                continue
            _, r, te, _, _ = oracles[i].step(a[i])
            e = oracles[i].sim.ego
            ref = np.array([e.x, e.y, e.yaw, e.v], dtype=np.float64)
            rel = np.abs(hero[i, :4] - ref) / np.maximum(np.abs(ref), 1.0)
            worst = max(worst, float(rel.max()))
            assert rel.max() < 1e-7, (t, i, hero[i, :4], ref)
            assert te == term[i] and abs(r - rew[i]) < 1e-9, (t, i)
            steps_alive[i] += 1
            alive[i] = not te
        if t in (250, 999):
            ego, act = eng.get_state(16)
            fov = eng.fov().cpu().numpy()
            for i in range(n):
                if alive[i]:
                    ref = np.array([[b.x, b.y, b.yaw, b.v] for b in oracles[i].sim.actors])
                    assert np.allclose(act[i, :len(ref), :4], ref, rtol=1e-7, atol=1e-7), (t, i, "actors")
                    assert np.array_equal(fov[i], oracles[i].render_index()), (t, i, "frame")
    assert steps_alive.max() == 1000 and (steps_alive >= 900).sum() >= 2, steps_alive
    print(f"max relative pose deviation over {steps_alive.tolist()} steps: {worst:.3e}")
    eng.close()


def test_step_host_matches_device_step():
    """cbev_step_host (pinned host actions in, reward / flags out on a side stream overlapped with the raster
    kernel) returns exactly what cbev_step leaves on the device."""
    import torch

    from carlabev_env_b200 import engine as E

    scenes = _scenes([("lead_brake", 1 + i % 3) for i in range(16)], seed0=700)
    n = 64
    a_dev = _engine(n, scenes, autoreset=E.AUTORESET_NEXT_STEP, seed=3)
    a_host = _engine(n, scenes, autoreset=E.AUTORESET_NEXT_STEP, seed=3)
    ids = torch.arange(n, dtype=torch.int32) % len(scenes)
    a_dev.reset(ids)
    a_host.reset(ids)
    out = torch.zeros(n * 10, dtype=torch.uint8).pin_memory()
    rew, term, trunc = out[: n * 8].view(torch.float64), out[n * 8: n * 9], out[n * 9:]
    sep = [torch.zeros(n, dtype=torch.float64).pin_memory(), torch.zeros(n, dtype=torch.uint8).pin_memory(),
           torch.zeros(n, dtype=torch.uint8).pin_memory()]
    g = torch.Generator().manual_seed(1)
    n_term = 0
    for t in range(60):
        a = torch.rand(n, 3, generator=g)
        a[:, 1] = a[:, 1] * 2 - 1
        ap = a.pin_memory()
        a_dev.step(a.cuda())
        if t % 2 == 0:
            a_host.step_host(ap, rew, term, trunc)          # contiguous outputs: single copy
            got = (rew, term, trunc)
        else:
            a_host.step_host(ap, *sep)                       # separate buffers: three copies
            got = sep
        torch.cuda.current_stream().synchronize()
        assert torch.equal(got[0], a_dev.reward.cpu()) and torch.equal(got[1], a_dev.terminated.cpu())
        assert torch.equal(got[2], a_dev.truncated.cpu())
        assert torch.equal(a_host.obs(), a_dev.obs())
        n_term += int(got[1].sum())
    assert n_term > 0
    a_dev.close()
    a_host.close()


def test_vector_env_temporal_fusion_and_mask_shapes():
    import torch

    from carlabev_env_b200 import EnvConfig, RunConfig, make_env

    scenes = _scenes([("lead_brake", 3)] * 2, seed0=77)
    for mode, c_out in (("vehicle_temporal", 8), ("vehicle_weighted", 6)):
        cfg = RunConfig(env=EnvConfig(action_mode="continuous", temporal_fusion_mode=mode, fov_masked=True), num_envs=2)
        envs = make_env(cfg, scenes=scenes, ring_budget_bytes=32 << 20)
        assert envs.single_observation_space.shape == (c_out, 96, 96)
        obs, _ = envs.reset(options={"scene_ids": np.arange(2)})
        assert obs.shape == (2, c_out, 96, 96)
        obs, *_ = envs.step(np.tile(np.array([[0.5, 0.0, 0.0]], np.float32), (2, 1)))
        assert obs.shape == (2, c_out, 96, 96) and float(obs.max()) <= 1.0
        assert float(obs[:, :, 0, 0].abs().sum()) == 0.0   # masked corner pixel matches no class
        envs.close()


def test_make_env_spaces_like_reference_smoke_tests():
    """The reference's tests/test_public_config.py:212-256: discrete9 -> Discrete(9), continuous -> Box shape (3,)."""
    from carlabev_env_b200 import EnvConfig, RunConfig, make_env

    scenes = _scenes([("lead_brake", 1)])
    envs = make_env(RunConfig(env=EnvConfig(), num_envs=1), scenes=scenes, ring_budget_bytes=16 << 20)
    assert envs.single_action_space.n == 9 and envs.single_observation_space.shape == (24, 96, 96)
    envs.close()
    envs = make_env(EnvConfig(action_mode="continuous", obs_mode="bev_rgb"), scenes=scenes, ring_budget_bytes=16 << 20)
    assert envs.single_action_space.shape == (3,) and envs.single_observation_space.shape == (4, 96, 96)
    assert envs.single_observation_space.dtype == np.uint8
    obs, _ = envs.reset(options={"scene_ids": 0})
    assert tuple(obs.shape) == (1, 4, 96, 96)
    envs.close()


def test_authored_scenes_pool_parity():
    """The reference's authored scene files (assets/scenes/*.json, incl. traffic lights and timed_brake /
    cross / stop_mid / yield_return behaviours), exported as a pool: every entry stepped against the oracle."""
    import torch

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.pool import load_shipped_pool, pack_pool
    from oracle.env import OracleEnv

    scenes = load_shipped_pool("authored_scenes")
    n = len(scenes)
    eng = E.Engine(n, obs_mode=E.OBS_SEMANTIC, mask_mode="7-class", frame_stack=4, action_mode=E.ACTION_CONTINUOUS,
                   max_actors=4, ring_budget_bytes=128 << 20)
    eng.upload_map(load_map())
    eng.upload_pool(pack_pool(scenes))
    oracles = [OracleEnv(load_map(), semantic_mask_ch="7-class", action_mode="continuous") for _ in range(n)]
    obs = eng.reset(torch.arange(n, dtype=torch.int32)).cpu().numpy()
    for i in range(n):
        assert np.array_equal(obs[i], oracles[i].reset(scenes[i]))
    rng = np.random.default_rng(8)
    alive = np.ones(n, bool)
    for t in range(70):
        a = _rand_actions(rng, n)
        a[:, 0] *= 0.4
        a[:, 1] *= 0.3
        if t < 30:
            a[::2] = np.array([0.0, 0.0, 1.0], np.float32)  # half of the envs wait so pedestrians / brakes play out
        eng.step(torch.from_numpy(a).cuda())
        obs, rew = eng.obs().cpu().numpy(), eng.reward.cpu().numpy()
        term, hero = eng.terminated.cpu().numpy().astype(bool), eng.hero.cpu().numpy()
        for i in range(n):
            if alive[i]:
                _check_env(t, i, hero[i], rew[i], term[i], obs[i], oracles[i], oracles[i].step(a[i]))
                alive[i] = not term[i]
    eng.close()


@pytest.mark.parametrize("anchor", [(0.5, 0.5), (0.5, 0.75), (0.5, 0.2)])
def test_raster_parity_over_all_headings(anchor):
    """Frames against the oracle for 384 ego headings per camera anchor (exact multiples of 45 degrees, their
    float neighbours, and a dense sweep): exercises the exact rotate90 path, the branch-free fast path and the
    generic path with pygame's range tests / background colour of the 16.16 fixed-point walk."""
    import torch

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.pool import load_shipped_pool, pack_pool
    from oracle import raster
    from oracle.env import OracleEnv

    scene = load_shipped_pool("rdm_rt_medium_v1")[3]
    special = [k * np.pi / 4 for k in range(-4, 4)]
    yaws = special + [np.nextafter(y, 10.0) for y in special] + [np.nextafter(y, -10.0) for y in special]
    yaws += list(np.linspace(-np.pi, np.pi, 384 - len(yaws), endpoint=False))
    n = len(yaws)
    eng = E.Engine(n, obs_mode=E.OBS_SEMANTIC, mask_mode="6-class", frame_stack=2, action_mode=E.ACTION_CONTINUOUS,
                   max_actors=16, anchor=anchor, ring_budget_bytes=256 << 20)
    eng.upload_map(load_map())
    eng.upload_pool(pack_pool([scene]))
    eng.keep_fov(True)
    eng.reset(torch.zeros(n, dtype=torch.int32))
    ego, _ = eng.get_state(16)
    ego[:, 2] = yaws            # yaw
    ego[:, 6] = yaws            # previous yaw
    ego[:, 3] = 0.0             # standing still: the heading is kept by the step
    eng.set_ego_state(ego)
    a = np.tile(np.array([[0.0, 0.0, 1.0]], np.float32), (n, 1))
    eng.step(torch.from_numpy(a).cuda())
    fov = eng.fov().cpu().numpy()
    obs = eng.obs().cpu().numpy()
    geom = raster.FovGeometry(128, *anchor)
    n_generic = 0
    for i, yaw in enumerate(yaws):
        o = OracleEnv(load_map(), action_mode="continuous", frame_stack=2, anchor=anchor)
        o.reset(scene)
        o.sim.ego.yaw = o.sim.ego.yaw_1 = float(yaw)
        o.sim.ego.v = 0.0
        ref_obs, *_ = o.step(a[i])
        assert float(o.sim.ego.yaw) == float(eng.hero[i, 2]), (i, yaw)
        ref = o.render_index()
        assert np.array_equal(fov[i], ref), (i, yaw, int((fov[i] != ref).sum()))
        assert np.array_equal(obs[i, 6:], ref_obs[6:]), (i, yaw)
        # does this heading leave the fast path? (window corners outside the rotated surface / source range)
        rp = raster.rotate_params(float(o.sim.ego.yaw), geom.crop)
        if rp["mode"] == 1:
            left, top = geom.anchor[0] - (rp["nx"] >> 1), geom.anchor[1] - (rp["ny"] >> 1)
            inside = left <= 0 and top <= 0 and left + rp["nx"] >= 128 and top + rp["ny"] >= 128
            for cx in (0, 127):
                for cy in (0, 127):
                    rxp, ryp = cx - left, cy - top
                    dx = rp["ax"] + rp["isin"] * (rp["cy"] - ryp) + rp["xd"] + rxp * rp["icos"]
                    dy = rp["ay"] - rp["icos"] * (rp["cy"] - ryp) + rp["yd"] + rxp * rp["isin"]
                    inside = inside and 0 <= dx <= (geom.crop << 16) - 1 and 0 <= dy <= (geom.crop << 16) - 1
            n_generic += not inside
    print(f"anchor {anchor}: {n} headings, {n_generic} on the generic (range-tested) path")
    eng.close()


def test_frame_recorder_env0(tmp_path):
    """capture_video: env 0's RGB field of view after reset and after every step of the selected episodes
    (RecordVideo's role in wrap_env, envs/__init__.py:40-60), checked against the oracle's frames."""
    from carlabev_env_b200 import RunConfig, EnvConfig, make_env
    from oracle import raster
    from oracle.env import OracleEnv

    scenes = _scenes([("lead_brake", 1), ("jaywalk", 2)])
    cfg = RunConfig(env=EnvConfig(obs_mode="bev_semantic", action_mode="continuous"), num_envs=2, capture_video=True,
                    video_output_dir=str(tmp_path), video_episode_indices=[0, 1], video_name_prefix="t")
    envs = make_env(cfg, scenes=scenes)
    ora = OracleEnv(load_map(), action_mode="continuous")
    ora.reset(scenes[0])
    want = [[ora.last_rgb]]
    envs.reset(options={"scene_ids": np.array([0, 0])})       # twin envs: both finish on the same step
    act = np.array([[1.0, 0.0, 0.0], [1.0, 0.0, 0.0]], np.float32)
    for ep in range(2):
        for _ in range(400):
            _, _, term, trunc, _ = envs.step(act)
            _, _, o_term, o_trunc, _ = ora.step(act[0])
            want[-1].append(ora.last_rgb)
            if bool(term[0] | trunc[0]):
                assert o_term or o_trunc
                break
        else:
            raise AssertionError("episode did not end")
        if ep == 0:
            envs.reset(options={"scene_ids": np.array([0, 0]), "reset_mask": (term | trunc).cpu().numpy()})
            ora.reset(scenes[0])
            want.append([ora.last_rgb])
    envs.close()
    files = sorted(os.listdir(tmp_path))
    assert files == ["t-episode-0.npy", "t-episode-1.npy"]
    for f, w in zip(files, want):
        got = np.load(os.path.join(tmp_path, f))
        assert got.shape == (len(w), 128, 128, 3) and got.dtype == np.uint8
        assert np.array_equal(got, np.stack(w))


@pytest.mark.parametrize("obs_size,mode", [((84, 84), "semantic"), ((64, 64), "semantic"), ((128, 128), "semantic"),
                                           ((112, 100), "semantic"), ((84, 84), "gray"), ((64, 64), "gray"),
                                           ((48, 64), "gray"), ((32, 32), "semantic"), ((160, 160), "semantic"),
                                           ((96, 144), "gray"), ((144, 96), "semantic"), ((48, 48), "semantic"),
                                           ((48, 48), "gray")])
def test_other_observation_sizes(obs_size, mode):
    """EnvConfig.obs_size other than (96, 96): ResizeObservation through OpenCV's area tables (float32, OpenCV's
    accumulation order), its 2x2 integer path for (64, 64), the plain copy for (128, 128), and its 8-bit bilinear
    kernel on area-mode coefficients as soon as one axis enlarges -- bit-exact masks /
    gray levels against the oracle (itself pinned on cv2 for these sizes).  (48, 48) is the 8 : 3 ratio: single-colour
    8 x 8 blocks leave from the registers of the rotate (k_render_any's block shortcut)."""
    import torch

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.pool import load_shipped_pool
    from oracle.env import OracleEnv

    scenes = _scenes([("lead_brake", 3), ("jaywalk", 4), ("jaywalk", 3)], seed0=1300) + load_shipped_pool("rdm_rt_medium_v1")[:3]
    n = len(scenes)
    gray = mode == "gray"
    eng = _engine(n, scenes, obs_size=obs_size, max_actors=20, obs_mode=E.OBS_GRAY if gray else E.OBS_SEMANTIC,
                  mask_mode="7-class")
    oracles = [OracleEnv(load_map(), action_mode="continuous", obs_size=obs_size, semantic_mask_ch="7-class",
                         obs_mode="bev_rgb" if gray else "bev_semantic") for _ in range(n)]
    obs = eng.reset(torch.arange(n, dtype=torch.int32)).cpu().numpy()
    C = 4 if gray else 4 * 7
    assert obs.shape == (n, C, *obs_size)
    for i in range(n):
        assert np.array_equal(obs[i], oracles[i].reset(scenes[i])), (i, "reset")
    rng = np.random.default_rng(5)
    alive = np.ones(n, bool)
    for t in range(30):
        a = _rand_actions(rng, n)
        eng.step(torch.from_numpy(a).cuda())
        obs = eng.obs().cpu().numpy()
        for i in range(n):
            if alive[i]:
                o, _, te, tr, _ = oracles[i].step(a[i])
                assert np.array_equal(obs[i], o), (t, i)
                alive[i] = not (te or tr)
    if not gray:  # the fusion kernel follows the observation size too
        from oracle import raster

        obs = eng.obs().cpu().numpy().reshape(n, 4, 7, *obs_size)
        for name, fn in (("vehicle_temporal", raster.fuse_vehicle_temporal), ("vehicle_weighted", raster.fuse_vehicle_weighted)):
            got = eng.fuse(name).cpu().numpy()
            for i in range(n):
                assert np.array_equal(got[i], fn(obs[i], "7-class")), (name, i)
    eng.close()


def test_observation_size_errors():
    from carlabev_env_b200 import engine as E

    scenes = _scenes([("lead_brake", 1)])
    for bad in [(96, 300), (4, 4), (50, 51)]:
        with pytest.raises(E.CbevError):
            _engine(1, scenes, obs_size=bad)


def test_sharded_vector_env_equals_the_slice_of_the_full_one():
    """make_env(cfg, shard=(rank, world)): the shard's envs are envs [lo, hi) of the unsharded VectorEnv
    (same per-env scene seeds, hence the same observations and rewards)."""
    from carlabev_env_b200 import EnvConfig, RunConfig, make_env

    cfg = RunConfig(env=EnvConfig(action_mode="continuous"), num_envs=6)
    opts = {"scene": "lead_brake", "level": 2}
    full = make_env(cfg, ring_budget_bytes=32 << 20)
    obs_full, _ = full.reset(seed=100, options=dict(opts))
    act = np.tile(np.array([[0.6, 0.1, 0.0]], np.float32), (6, 1))
    _, rew_full, *_ = full.step(act)
    for rank in range(3):
        part = make_env(cfg, shard=(rank, 3), ring_budget_bytes=32 << 20)
        assert part.num_envs == 2 and part.env_offset == 2 * rank
        obs, _ = part.reset(seed=100, options=dict(opts))
        assert bool((obs == obs_full[2 * rank: 2 * rank + 2]).all())
        _, rew, *_ = part.step(act[:2])
        assert bool((rew == rew_full[2 * rank: 2 * rank + 2]).all())
        part.close()
    full.close()
    with pytest.raises(ValueError):
        make_env(cfg, shard=(0, 4))


@pytest.mark.parametrize("seed", [3, 6, 27, 30])
def test_random_configurations_against_the_oracle(seed):
    """Random env configuration (action profile, reward mode, mask channels, camera anchor, fov mask, gray /
    semantic), host-generated scenes of every kind and random actions: engine == oracle on observations, rewards,
    flags and poses.  The same generator drives oracle/fuzz_steps.py against the unmodified reference."""
    import torch

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200 import scenes as S
    from carlabev_env_b200.config import ACTION_PROFILES
    from carlabev_env_b200.fovmask import corner_mask
    from carlabev_env_b200.pool import pack_pool
    from oracle.env import OracleEnv

    rng = np.random.default_rng(seed)
    cls = load_map()
    profile = str(rng.choice(["continuous_gsb_v1", "discrete9_v1", "discrete13_v1"]))
    continuous = profile == "continuous_gsb_v1"
    reward = "shaping" if rng.random() < 0.4 else "carl"
    mask = str(rng.choice(["6-class", "7-class", "5-class", "4-class", "binary"]))
    anchor = (0.5, 0.75) if rng.random() < 0.4 else (0.5, 0.5)
    fov_masked = bool(rng.random() < 0.4)
    gray = bool(rng.random() < 0.3)
    pad = 230 if anchor[1] == 0.75 else 182
    reqs = [dict(scene="rdm", num_vehicles=int(rng.integers(0, 9)), route_dist_range=[30, 90], scene_seed=int(rng.integers(0, 10**6)))
            for _ in range(5)]
    reqs += [dict(scene="lead_brake", level=int(rng.integers(1, 4)), scene_seed=int(rng.integers(0, 10**6))) for _ in range(3)]
    reqs += [dict(scene="jaywalk", level=int(rng.integers(1, 5)), scene_seed=int(rng.integers(0, 10**6))) for _ in range(3)]
    reqs += [dict(scene="red_light_runner", scene_seed=int(rng.integers(0, 10**6)))]
    scenes = [S.build_scene(r, cls_map=cls, pad=pad) for r in reqs]
    n = len(scenes)
    eng = E.Engine(n, obs_mode=E.OBS_GRAY if gray else E.OBS_SEMANTIC, mask_mode=mask, frame_stack=4,
                   action_mode=E.ACTION_CONTINUOUS if continuous else E.ACTION_DISCRETE,
                   discrete_table=ACTION_PROFILES[profile].get("discrete_actions"),
                   reward_mode=E.REWARD_SHAPING if reward == "shaping" else E.REWARD_CARL, anchor=anchor, max_actors=12,
                   ring_budget_bytes=64 << 20)
    eng.upload_map(cls)
    eng.upload_pool(pack_pool(scenes))
    if fov_masked:
        eng.upload_fov_mask(corner_mask(128, 0.5))
    oracles = [OracleEnv(cls, obs_mode="bev_gray" if gray else "bev_semantic", semantic_mask_ch=mask,
                         action_mode="continuous" if continuous else "discrete", action_profile=profile,
                         reward_mode=reward, anchor=anchor, fov_masked=fov_masked) for _ in range(n)]
    obs = eng.reset(torch.arange(n, dtype=torch.int32)).cpu().numpy()
    for i in range(n):
        assert np.array_equal(obs[i], oracles[i].reset(scenes[i])), (i, "reset")
    alive = np.ones(n, bool)
    n_act = len(ACTION_PROFILES[profile].get("discrete_actions") or [])
    for t in range(40):
        if continuous:
            a = _rand_actions(rng, n)
            a[:, 2] *= rng.random(n) < 0.2
            dev_a = torch.from_numpy(a).cuda()
        else:
            a = rng.integers(0, n_act, n)
            dev_a = torch.from_numpy(a).cuda()
        eng.step(dev_a)
        obs, rew = eng.obs().cpu().numpy(), eng.reward.cpu().numpy()
        term, trunc = eng.terminated.cpu().numpy().astype(bool), eng.truncated.cpu().numpy().astype(bool)
        hero = eng.hero.cpu().numpy()
        for i in range(n):
            if not alive[i]:
                continue
            o, r, te, tr, _ = oracles[i].step(a[i] if continuous else int(a[i]))
            e = oracles[i].sim.ego
            assert np.array_equal(obs[i], o), (t, i, reqs[i], "observation")
            assert abs(r - rew[i]) < 1e-9 and te == term[i] and tr == trunc[i], (t, i, reqs[i], r, rew[i])
            assert np.allclose(hero[i, :4], [e.x, e.y, e.yaw, e.v], rtol=1e-9, atol=1e-9), (t, i, "pose")
            alive[i] = not (te or tr)
    eng.close()


def test_bench_dump_outputs_repeat_and_follow_steps(tmp_path):
    """bench.py --dump-outputs: the same arguments give the same arrays bit for bit (two builds can be compared output
    for output), every array is float32 / float64 and all fit in 64 MB, and --steps sets how far the state has moved."""
    import subprocess
    import sys

    from golden_util import ROOT

    def run(tag, steps):
        out = tmp_path / tag
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                            "--warmup", "3", "--envs", "512", "--pool", "64", "--no-extras", "--no-cpu-baseline",
                            "--dump-outputs", str(out)], env={**os.environ, "TMPDIR": str(tmp_path)},
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        return {f[:-len(".npy")]: np.load(out / f) for f in sorted(os.listdir(out))}

    a, b, c = run("a", 7), run("b", 7), run("c", 8)
    assert sorted(a) == ["cause", "env_ids", "episode", "hero", "obs", "obs_env_ids", "reward", "terminated", "truncated"]
    assert a["obs"].shape[1:] == (24, 96, 96) and a["reward"].shape == (512,) and a["hero"].shape[0] == 512
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        assert np.array_equal(a[k], b[k], equal_nan=True), k
    assert not np.array_equal(a["hero"], c["hero"])


def test_bench_dump_rows_are_the_engine_outputs_of_the_named_envs(tmp_path, monkeypatch):
    """bench.dump_outputs on a subset of the envs: row j of every per-env file is env env_ids[j] of the engine, row j of
    obs.npy is the observation window of env obs_env_ids[j]."""
    import torch

    import bench
    from carlabev_env_b200 import engine as E

    n = 96
    eng = _engine(n, _scenes([("lead_brake", 1 + i % 3) for i in range(12)], seed0=700),
                  autoreset=E.AUTORESET_NEXT_STEP, seed=3)
    eng.reset(torch.arange(n, dtype=torch.int32) % 12)
    rng = np.random.default_rng(4)
    for _ in range(30):
        eng.step(torch.from_numpy(_rand_actions(rng, n)).cuda())
    monkeypatch.setattr(bench, "DUMP_ENVS", 40)
    monkeypatch.setattr(bench, "DUMP_OBS_BYTES", 7 * 24 * 96 * 96 * 4)
    bench.dump_outputs(str(tmp_path), eng)
    d = {k: np.load(tmp_path / f"{k}.npy") for k in ("env_ids", "obs_env_ids", "reward", "terminated", "truncated",
                                                    "cause", "hero", "episode", "obs")}
    ids, obs_ids = d["env_ids"].astype(np.int64), d["obs_env_ids"].astype(np.int64)
    assert len(ids) == 40 == len(set(ids.tolist())) and len(obs_ids) == 7 and ids.max() < n and obs_ids.max() < n
    assert ids.tolist() != list(range(40))   # a seeded sample, not the first envs
    for k in ("reward", "hero", "episode"):
        assert np.array_equal(d[k], getattr(eng, k).cpu().numpy()[ids]), k
    for k in ("terminated", "truncated", "cause"):
        assert np.array_equal(d[k], getattr(eng, k).cpu().numpy()[ids].astype(np.float32)), k
    assert np.array_equal(d["obs"], eng.obs().cpu().numpy()[obs_ids])
    assert d["terminated"].any() or d["reward"].std() > 0   # the rows carry data, not zeros
    eng.close()

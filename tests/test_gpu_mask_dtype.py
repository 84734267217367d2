"""uint8 semantic masks (mask_dtype="uint8", CBEV_OBS_SEMANTIC_U8) on the GPU: a float32 and a uint8 engine with the
same configuration, pool, seed and actions (device auto-reset on) must agree bit for bit at every step -- the uint8
window equals the float32 window cast to uint8, the float32 window holds only 0 and 1, and rewards, flags, hero and
episode blocks are identical.  Covers every mask mode through k_render, every resize branch of k_render_any, the
oracle directly, both fusion modes, the make_env surface and the benchmark scale."""
import numpy as np
import pytest

from golden_util import load_map

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

MASKS = ("binary", "2-class", "4-class", "5-class", "6-class", "7-class")


def _scripted(n, seed0=500):
    from carlabev_env_b200.scenes import build_scripted_scene

    cls = load_map()
    kinds = [("lead_brake", 1 + i % 3) if i % 2 == 0 else ("jaywalk", 1 + i % 4) for i in range(n)]
    return [build_scripted_scene(k, seed0 + i, level=lv, cls_map=cls) for i, (k, lv) in enumerate(kinds)]


def _rdm(size, n=24):
    from carlabev_env_b200.scenes import build_pool

    pad = {64: 91, 128: 182, 256: 363}[size]
    return [s for s in build_pool([dict(scene="rdm", num_vehicles=12, route_dist_range=(30, 100), scene_seed=i)
                                   for i in range(n)], pad=pad, size=size, skip_invalid=True) if s is not None]


def _same_masks(f32, u8, what):
    import torch

    assert f32.dtype == torch.float32 and u8.dtype == torch.uint8, what
    assert f32.shape == u8.shape, what
    assert bool(((f32 == 0) | (f32 == 1)).all()), (what, "float masks are not 0 / 1")
    assert torch.equal(u8, f32.to(torch.uint8)), (what, int((u8 != f32.to(torch.uint8)).sum()))


def _same_outputs(engs, what):
    import torch

    f, u = engs
    for name in ("reward", "terminated", "truncated", "cause", "hero"):
        assert torch.equal(getattr(f, name), getattr(u, name)), (what, name)
    assert np.array_equal(f.episode.cpu().numpy(), u.episode.cpu().numpy(), equal_nan=True), (what, "episode")


def _run_pair(scenes, n=64, steps=60, mask_mode="6-class", ring_slots=8, size=128, obs_size=(96, 96), flags=0,
              partial_reset_at=None, max_actors=16):
    """Both dtypes side by side; returns the number of terminal env-steps seen (each is followed by a reset frame)."""
    import torch

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.pool import pack_pool

    engs = []
    for dt in ("float32", "uint8"):
        e = E.Engine(n, mask_mode=mask_mode, frame_stack=4, ring_slots=ring_slots, action_mode=E.ACTION_CONTINUOUS,
                     autoreset=E.AUTORESET_NEXT_STEP, max_actors=max_actors, size=size, obs_size=obs_size, seed=3,
                     mask_dtype=dt)
        e.upload_map(load_map(size))
        e.upload_pool(pack_pool(scenes))
        e.set_debug_flags(flags)
        engs.append(e)
    assert engs[1].frame_bytes * 4 == engs[0].frame_bytes
    ids = torch.arange(n, dtype=torch.int32) % len(scenes)
    obs = [e.reset(ids) for e in engs]
    _same_masks(*obs, "reset")
    assert obs[0].any()
    rng = np.random.default_rng(size + obs_size[0] + flags)
    done = 0
    for t in range(steps):
        a = np.stack([rng.uniform(0, 1, n), rng.uniform(-1, 1, n), rng.uniform(0, 1, n)], axis=1).astype(np.float32)
        a = torch.from_numpy(a).cuda()
        for e in engs:
            e.step(a)
        _same_masks(engs[0].obs(), engs[1].obs(), (t, "step"))
        _same_outputs(engs, t)
        done += int((engs[0].terminated | engs[0].truncated).sum())
        if t == partial_reset_at:
            mask = torch.arange(n) % 3 == 0
            obs = [e.reset((ids + 5) % len(scenes), mask) for e in engs]
            _same_masks(*obs, (t, "masked reset"))
    for e in engs:
        e.close()
    return done


@pytest.mark.parametrize("mask_mode", MASKS)
def test_every_mask_mode_through_k_render(mask_mode):
    """k_render (size 128 / (96, 96)): reset frames from device auto-reset, a masked partial reset, and ring_slots 7
    and 9 so that the mirror write and the wrap of the ring are both crossed."""
    scenes = _scripted(16)
    ring_slots = 7 if MASKS.index(mask_mode) % 2 == 0 else 9
    done = _run_pair(scenes, mask_mode=mask_mode, ring_slots=ring_slots, partial_reset_at=20, max_actors=4)
    assert done > 0


@pytest.mark.parametrize("size,obs_size,flags", [
    (64, (96, 96), 0),      # an axis enlarges: bilinear
    (256, (96, 96), 0),     # table resize with the 8 : 3 block shortcut
    (256, (96, 96), 512),   # table resize without it
    (128, (84, 84), 0),     # table resize
    (128, (64, 64), 0),     # exact halving
    (128, (128, 128), 0),   # copy
    (128, (96, 96), 256),   # the k_render configuration through k_render_any
    (128, (96, 96), 1),     # k_render with the generic (range-tested) rotate
    (128, (84, 84), 1),     # k_render_any with the generic rotate
])
def test_every_resize_branch_of_k_render_any(size, obs_size, flags):
    scenes = _rdm(size)
    assert len(scenes) >= 8
    _run_pair(scenes, steps=40, size=size, obs_size=obs_size, flags=flags, partial_reset_at=15)


def test_uint8_masks_against_the_oracle():
    """As test_batched_parity_with_masked_resets, with the uint8 engine: lead_brake and jaywalk, masked resets."""
    import torch

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.pool import pack_pool
    from oracle.env import OracleEnv

    scenes = _scripted(20)
    n = len(scenes)
    eng = E.Engine(n, mask_mode="6-class", frame_stack=4, action_mode=E.ACTION_CONTINUOUS, max_actors=4,
                   ring_budget_bytes=16 << 20, mask_dtype="uint8")
    eng.upload_map(load_map())
    eng.upload_pool(pack_pool(scenes))
    oracles = [OracleEnv(load_map(), action_mode="continuous") for _ in range(n)]
    scene_of = np.arange(n)
    obs = eng.reset(torch.arange(n, dtype=torch.int32)).cpu().numpy()
    assert obs.dtype == np.uint8 and obs.shape == (n, 24, 96, 96)
    for i in range(n):
        assert np.array_equal(obs[i], oracles[i].reset(scenes[i])), (i, "reset")
    rng = np.random.default_rng(1)
    n_resets = 0
    for t in range(60):
        a = np.stack([rng.uniform(0, 1, n), rng.uniform(-1, 1, n), rng.uniform(0, 1, n)], axis=1).astype(np.float32)
        eng.step(torch.from_numpy(a).cuda())
        obs, rew = eng.obs().cpu().numpy(), eng.reward.cpu().numpy()
        term = eng.terminated.cpu().numpy().astype(bool)
        for i in range(n):
            o, r, te, _, _ = oracles[i].step(a[i])
            assert np.array_equal(obs[i], o), (t, i, "observation")
            assert abs(r - rew[i]) < 1e-9 and te == term[i], (t, i, "reward / terminated")
        if term.any():
            scene_of[term] = (scene_of[term] + 7) % n
            obs = eng.reset(torch.from_numpy(scene_of.astype(np.int32)), term).cpu().numpy()
            for i in np.flatnonzero(term):
                assert np.array_equal(obs[i], oracles[i].reset(scenes[scene_of[i]])), (t, i, "masked reset")
                n_resets += 1
    assert n_resets > 0
    eng.close()


def _env_pair(scenes, n, fusion="stack", mask_ch="6-class", **kw):
    from carlabev_env_b200 import EnvConfig, RunConfig, make_env

    cfg = RunConfig(env=EnvConfig(action_mode="continuous", temporal_fusion_mode=fusion, semantic_mask_ch=mask_ch),
                    num_envs=n)
    return [make_env(cfg, scenes=scenes, autoreset="next_step", ring_slots=8, mask_dtype=dt, **kw)
            for dt in ("float32", "uint8")]


@pytest.mark.parametrize("mask_ch", ["4-class", "7-class"])
def test_fusion_through_make_env(mask_ch):
    """vehicle_temporal on a uint8 ring gives uint8 equal to the float fused output; vehicle_weighted on a uint8 ring is
    float32 bit-identical to the float path."""
    import torch

    scenes = _scripted(8)
    n = 16
    for fusion in ("vehicle_temporal", "vehicle_weighted"):
        envs = _env_pair(scenes, n, fusion, mask_ch)
        outs = [e.reset(options={"scene_ids": np.arange(n) % len(scenes)})[0] for e in envs]
        rng = np.random.default_rng(5)
        seen_weighted = False
        for t in range(40):
            if fusion == "vehicle_temporal":
                _same_masks(*outs, (fusion, t))
            else:
                assert outs[0].dtype == outs[1].dtype == torch.float32
                assert torch.equal(outs[0], outs[1]), (fusion, t)
                seen_weighted |= bool(((outs[1] > 0) & (outs[1] < 1)).any())
            a = np.stack([rng.uniform(0.3, 1, n), rng.uniform(-0.3, 0.3, n), rng.uniform(0, 0.1, n)], axis=1).astype(np.float32)
            outs = [e.step(a)[0] for e in envs]
        if fusion == "vehicle_weighted":
            assert seen_weighted, "no fractional vehicle history was produced"
        for e in envs:
            e.close()


def test_make_env_surface():
    import torch

    from carlabev_env_b200 import EnvConfig, RunConfig, make_env

    scenes = _scripted(8)
    n = 8
    for fusion, c_out, dtype in (("stack", 24, np.uint8), ("vehicle_temporal", 8, np.uint8),
                                 ("vehicle_weighted", 6, np.float32)):
        cfg = RunConfig(env=EnvConfig(action_mode="continuous", temporal_fusion_mode=fusion), num_envs=n)
        envs = make_env(cfg, scenes=scenes, ring_budget_bytes=16 << 20, mask_dtype="uint8", to_numpy=True)
        sp = envs.single_observation_space
        assert sp.shape == (c_out, 96, 96) and np.dtype(sp.dtype) == np.dtype(dtype)
        assert float(np.min(sp.low)) == 0 and float(np.max(sp.high)) == 1
        obs, _ = envs.reset(options={"scene_ids": np.arange(n)})
        assert isinstance(obs, np.ndarray) and obs.dtype == dtype and obs.shape == (n, c_out, 96, 96)
        obs, *_ = envs.step(np.zeros((n, 3), np.float32))
        assert obs.dtype == dtype and sp.contains(obs[0])
        envs.close()
    # one auto-reset episode against the float32 make_env: observations, rewards, flags and terminal infos
    envs = _env_pair(scenes, n)
    outs = [e.reset(options={"scene_ids": np.arange(n)})[0] for e in envs]
    _same_masks(*outs, "reset")
    rng = np.random.default_rng(9)
    finished = None
    for t in range(400):
        a = np.stack([rng.uniform(0.5, 1, n), rng.uniform(-1, 1, n), rng.uniform(0, 0.1, n)], axis=1).astype(np.float32)
        res = [e.step(a) for e in envs]
        _same_masks(res[0][0], res[1][0], t)
        for k in (1, 2, 3):
            assert torch.equal(res[0][k], res[1][k]), (t, k)
        assert ("episode_info" in res[0][4]) == ("episode_info" in res[1][4])
        if "episode_info" in res[0][4]:
            for key in ("return", "length", "termination"):
                assert np.array_equal(res[0][4]["episode_info"][key], res[1][4]["episode_info"][key]), (t, key)
        if finished is not None and t == finished + 1:
            break  # the step that consumed the device auto-reset
        if finished is None and bool((res[0][2] | res[0][3]).any()):
            finished = t
    assert finished is not None
    for e in envs:
        e.close()


def test_benchmark_scale_c2():
    """The bench line's configuration (c2: 4096 envs, lead_brake, continuous actions, 6-class 96 x 96, F = 4, device
    auto-reset) for 120 steps: every env's window is equal between the two dtypes at every step."""
    import torch

    from carlabev_env_b200 import engine as E

    n, k = 4096, 1024
    engs = []
    for dt in ("float32", "uint8"):
        e = E.Engine(n, mask_mode="6-class", frame_stack=4, ring_slots=9, action_mode=E.ACTION_CONTINUOUS,
                     autoreset=E.AUTORESET_NEXT_STEP, max_actors=4, seed=11, mask_dtype=dt)
        e.upload_map(load_map())
        e.generate_scripted_pool(["lead_brake"] * k, [1 + i % 3 for i in range(k)], list(range(k)))
        engs.append(e)
    ids = torch.arange(n, dtype=torch.int32) % k
    _same_masks(*[e.reset(ids) for e in engs], "reset")
    g = torch.Generator(device="cuda")
    g.manual_seed(0)
    done = 0
    for t in range(120):
        a = torch.rand(n, 3, device="cuda", generator=g)
        a[:, 1] = 2 * a[:, 1] - 1
        for e in engs:
            e.step(a)
        _same_masks(engs[0].obs(), engs[1].obs(), t)
        _same_outputs(engs, t)
        done += int(engs[0].terminated.sum())
    assert done > 0
    for e in engs:
        e.close()

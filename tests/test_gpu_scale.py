"""Parity with the oracle AT THE BENCHMARK SIZES (BASELINE.json configs[1..3] per-GPU shapes): the engine runs
4096 / 8192 environments with device auto-reset exactly as `bench.py` drives it, and a seeded random sample of
64 environments is compared step for step with `OracleEnv` -- stacked observation, reward, flags, cause, all 32
hero fields, actor poses, the episode row of every terminal step, and the scene every auto-reset draws (replayed
through the same counter hash).  The whole statistics vector must equal the sum of the oracle's episode rows of the
compared envs and the engine's rows of the others; episode counter == number of terminal flags raised, step counter
== steps x N.

The step order compared is the reference's (envs/carlabev.py:223-231): scene step -> collision -> reward /
termination -> observation."""
import numpy as np
import pytest

from golden_util import load_map

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

M64 = (1 << 64) - 1
# Poses: the bar is 1e-5 relative after 1000 steps (BASELINE.json).  Live-stepped actors in closed-loop Stanley control
# amplify the 1-2 ulp differences between CUDA's and glibc's sincos / tan / atan2: 2e-9 was observed on a turning
# red_light_runner adversary after 76 steps; 1e-7 leaves two decades of margin to the bar.  Flags, rewards (1e-9) and
# every observation value stay exact.
POSE_TOL = 1e-7
# RETREAT NOTE.  A StopReturn pedestrian that turns back gets a NEW route, smoothed at that moment (jaywalk.py:43-54),
# made of its current position followed by the waypoints behind it.  When it stands short of the waypoint it was heading
# for, that route starts with a reversal: headings like [-2.86, -0.18, 0, 0] rad over points 1.5 px apart, which a
# bicycle model with a 2.9 px wheelbase cannot follow.  The closed loop is then CHAOTIC IN THE REFERENCE ITSELF: perturbing
# the smoothed retreat route by 1e-13 px in the oracle alone (the size of the difference between SciPy's LAPACK edge fit
# and the linear Savitzky-Golay operator the device applies -- and of BLAS-build differences) grows by ~2.4x per step
# to O(1) rad within ~60 steps in half of the level-3 scenes (measured, DESIGN.md section 2).  Nobody who does not
# reproduce LAPACK bit for bit can track such a pedestrian, so from the step a pedestrian switches to its retreat route
# the sampled env is FOLLOWED (episode boundaries taken from the engine) but not compared until its next reset; the
# fraction of such env-steps is bounded below.  The golden replay of a retreat (tests/golden/jaywalk_levels, a route
# without reversal) is exact to 1e-9 for its whole length.


def _splitmix64(z):
    z = (z + 0x9E3779B97F4A7C15) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def autoreset_scene(seed, env, episode, n_scenes):
    """sim.cu: device auto-reset draw of env `env` after its `episode`-th finished episode."""
    return _splitmix64((seed + env * 0x9E3779B97F4A7C15 + episode * 0xD1B54A32D192ED03) & M64) % n_scenes


# Hero fields by comparison bar (replay_golden's and the bars above): exact, pose-like, comfort.
HERO_EXACT = ("target_idx", "hit", "hit_id", "tile_class", "n_nearby", "scene", "cmd_gas", "cmd_steer", "cmd_brake", "t")
HERO_POSE = ("x", "y", "yaw", "v", "x_1", "y_1", "yaw_1", "v_1", "dist2wp", "set_point_x", "set_point_y",
             "set_point_yaw", "applied_delta", "acc", "dist2goal")
HERO_COMFORT = ("speed_mps", "accel_long", "accel_lat", "jerk_long", "jerk_lat", "yaw_rate", "yaw_acc")
EPISODE_EXACT = ("length", "cause", "scene", "num_vehicles", "episode")


def _field_index(fields, names):
    return np.array([fields.index(k) for k in names])


def _check_hero(got, ref, pose_tol, where):
    from carlabev_env_b200 import engine as E

    F = E.HERO_FIELDS
    assert sorted(HERO_EXACT + HERO_POSE + HERO_COMFORT) == sorted(F)
    for names, ok in ((HERO_EXACT, lambda g, r: g == r),
                      (HERO_POSE, lambda g, r: np.isclose(g, r, rtol=pose_tol, atol=pose_tol)),
                      (HERO_COMFORT, lambda g, r: np.isclose(g, r, rtol=1e-7, atol=1e-7))):
        c = _field_index(F, names)
        bad = np.flatnonzero(~ok(got[c], ref[c]))
        assert not len(bad), (*where, "hero", [(names[b], got[c[b]], ref[c[b]]) for b in bad])


def _check_episode(got, ref, where):
    """Counts and ids exact; means, return and len_ego_route to 1e-7 relative (replay_golden's bar)."""
    from carlabev_env_b200 import engine as E

    F = E.EPISODE_FIELDS
    c = _field_index(F, EPISODE_EXACT)
    assert np.array_equal(got[c], ref[c]), (*where, "episode", dict(zip(EPISODE_EXACT, zip(got[c], ref[c]))))
    bad = [k for k in F if k not in EPISODE_EXACT
           and abs(got[F.index(k)] - ref[F.index(k)]) > 1e-7 * max(1.0, abs(ref[F.index(k)]))]
    assert not bad, (*where, "episode", [(k, got[F.index(k)], ref[F.index(k)]) for k in bad])


def run_scale_parity(scenes, n_envs, *, steps, make_actions, engine_kw, oracle_kw, sample=64, seed=17,
                     min_autoresets=1, check_actors=True):
    """Engine vs oracle on `sample` envs of an `n_envs` batch (all of them when sample >= n_envs).  Per step and compared
    env: observation, reward, flags, cause, the whole hero block, actor poses, and the episode row on terminal steps;
    at the end the statistics vector against the sum of the compared envs' oracle episode rows plus the engine's rows
    of the others.  `make_actions(rng, n, t, hero)` gets the engine's hero block of the previous step (device tensor)
    and returns the actions of all n envs; the same action goes to both sides.  With autoreset=AUTORESET_DISABLED the
    envs that ended are reset by a masked `reset` after each step.  Returns (auto-resets, terminal steps, counts of
    the reward terms `oracle_pool.active_terms` saw active on compared env-steps)."""
    import torch

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.pool import pack_pool
    from oracle_pool import OraclePool
    from test_gpu_action_repeat import _stats_from_rows

    cls = load_map()
    K = len(scenes)
    amax = int(max(len(s["act_kind"]) for s in scenes))
    kw = dict(obs_mode=E.OBS_SEMANTIC, mask_mode="6-class", frame_stack=4, autoreset=E.AUTORESET_NEXT_STEP,
              max_actors=max(amax, 1), seed=seed, ring_budget_bytes=24 << 30)
    kw.update(engine_kw)
    next_step = kw["autoreset"] == E.AUTORESET_NEXT_STEP
    traj = int(kw.get("trajectory_steps", 1024))
    eng = E.Engine(n_envs, **kw)
    eng.upload_map(cls)
    eng.upload_pool(pack_pool(scenes))
    eng.reset(torch.arange(n_envs, dtype=torch.int32) % K)
    rng = np.random.default_rng(seed)
    if sample >= n_envs:
        idx = np.arange(n_envs, dtype=np.int64)
    else:  # the sample always holds the first / last env of the batch and of a CTA-sized block, the rest is random
        fixed = [0, 1, 15, 16, n_envs - 1]
        rest = rng.choice(np.setdiff1d(np.arange(n_envs), fixed), size=sample - len(fixed), replace=False)
        idx = np.sort(np.concatenate([fixed, rest])).astype(np.int64)
    idx_t = torch.from_numpy(idx).cuda()
    sampled = torch.zeros(n_envs, dtype=torch.bool, device="cuda")
    sampled[idx_t] = True
    pool = OraclePool(len(idx), scenes, oracle_kw)
    try:
        ref = pool.run([("reset", int(i) % K) for i in idx])
        obs0 = eng.obs()[idx_t].cpu().numpy()
        for j, i in enumerate(idx):
            assert np.array_equal(obs0[j], ref[j]["obs"]), (i, "reset observation")
        done = np.zeros(len(idx), bool)
        unpinned = np.zeros(len(idx), bool)   # see RETREAT NOTE: env is followed, not compared, until its next reset
        episodes = np.zeros(len(idx), dtype=np.int64)
        since_reset = np.zeros(len(idx), dtype=np.int64)
        n_auto = n_term = n_unpinned = 0
        term_total = torch.zeros((), dtype=torch.int64, device="cuda")
        rows = []      # what the statistics vector must add up to: one episode row per terminal env-step
        terms = {}     # reward terms active on compared env-steps
        for t in range(steps):
            a = make_actions(rng, n_envs, t, eng.hero)
            eng.step(torch.from_numpy(a).cuda())
            # the oracle sample steps on the host cores while the device works
            drawn = [autoreset_scene(seed, int(i), int(episodes[j]), K) if done[j] else -1 for j, i in enumerate(idx)]
            cmds = [("reset", drawn[j]) if done[j] else ("step", a[int(i)]) for j, i in enumerate(idx)]
            ref = pool.run(cmds)
            ended_all = (eng.terminated | eng.truncated).bool()
            term_total += eng.terminated.sum()
            # episode rows of the envs the oracle does not stand for; the compared ones add the oracle's row below
            rows.append(eng.episode[eng.terminated.bool() & ~sampled].cpu().numpy())
            obs = eng.obs()[idx_t].cpu().numpy()
            rew = eng.reward[idx_t].cpu().numpy()
            term = eng.terminated[idx_t].cpu().numpy().astype(bool)
            trunc = eng.truncated[idx_t].cpu().numpy().astype(bool)
            cause = eng.cause[idx_t].cpu().numpy()
            hero = eng.hero[idx_t].cpu().numpy()
            episode = eng.episode[idx_t].cpu().numpy()
            act = eng.get_state(amax)[1][idx] if check_actors and amax else None
            for j, i in enumerate(idx):
                i, r = int(i), ref[j]
                if done[j]:  # gymnasium NEXT_STEP: this step resets, ignores the action, reward 0, not terminated
                    assert np.array_equal(hero[j], r["hero"]), (t, i, "auto-reset hero block", hero[j], r["hero"])
                    assert rew[j] == 0.0 and not term[j] and not trunc[j] and cause[j] == 0, (t, i)
                    assert np.array_equal(obs[j], r["obs"]), (t, i, "auto-reset observation")
                    done[j] = False
                    unpinned[j] = False
                    since_reset[j] = 0
                    n_auto += 1
                    continue
                since_reset[j] += 1
                if unpinned[j]:
                    n_unpinned += 1
                    if term[j] or trunc[j]:   # follow the engine's episode boundary; both sides re-sync at the reset
                        if term[j]:
                            rows.append(episode[j][None])
                        done[j] = True
                        episodes[j] += 1
                        n_term += 1
                    continue
                # actor poses come from the exact tables until they run out, then from live (chaotic) stepping
                pose_tol = POSE_TOL if traj == 0 or since_reset[j] > traj else 1e-9
                assert abs(r["reward"] - rew[j]) < 1e-9, (t, i, "reward", r["reward"], rew[j])
                assert r["term"] == term[j] and r["trunc"] == trunc[j], (t, i, "flags")
                assert r["cause"] == cause[j], (t, i, "cause", r["cause"], cause[j])
                _check_hero(hero[j], r["hero"], pose_tol, (t, i))
                assert np.array_equal(obs[j], r["obs"]), (t, i, "observation", int((obs[j] != r["obs"]).sum()))
                if act is not None and len(r["actors"]):
                    na = len(r["actors"])
                    assert np.allclose(act[j, :na, :4], r["actors"], rtol=POSE_TOL, atol=POSE_TOL), (t, i, "actor poses")
                    if np.any(act[j, :na, 7].astype(np.int64) & 32):
                        unpinned[j] = True   # a pedestrian has just switched to a retreat route: RETREAT NOTE
                for k, on in r["terms"].items():
                    terms[k] = terms.get(k, 0) + int(on)
                if r["term"]:
                    _check_episode(episode[j], r["episode"], (t, i))
                    rows.append(r["episode"][None])
                if r["term"] or r["trunc"]:
                    done[j] = True
                    episodes[j] += 1
                    n_term += 1
            if not next_step and ended_all.any():  # SyncVectorEnv-style masked reset of every env that ended
                scene_ids = (torch.arange(n_envs, device="cuda") + 7 * (t + 1)) % K
                obs_r = eng.reset(scene_ids.to(torch.int32), ended_all)[idx_t].cpu().numpy()
                ids = scene_ids[idx_t].cpu().numpy()
                ref = pool.run([("reset", int(ids[j])) if done[j] else None for j in range(len(idx))])
                for j in np.flatnonzero(done):
                    assert np.array_equal(obs_r[j], ref[j]["obs"]), (t, int(idx[j]), "masked reset observation")
                unpinned[done] = False
                since_reset[done] = 0
                done[:] = False
    finally:
        pool.close()
    stats = eng.read_stats().cpu().numpy()
    assert stats[0] == int(term_total), "episode counter != number of terminal flags raised over the whole batch"
    assert stats[-1] == steps * n_envs
    want = _stats_from_rows(np.concatenate(rows) if rows else np.zeros((0, len(E.EPISODE_FIELDS))))
    counts = [0, 2] + list(range(4, 12))  # CBEV_S_EPISODES, the summed lengths and the per-cause counters
    assert np.array_equal(stats[counts], want[counts]), ("statistics counts", stats[counts], want[counts])
    sums = [c for c in range(len(stats) - 1) if c not in counts]
    assert np.allclose(stats[sums], want[sums], rtol=1e-7, atol=1e-7), ("statistics sums", stats[sums], want[sums])
    assert n_auto >= min_autoresets, (n_auto, n_term)
    assert n_unpinned <= 0.25 * steps * len(idx), f"{n_unpinned} of {steps * len(idx)} sampled env-steps were not compared"
    eng.close()
    return n_auto, n_term, terms


def _uniform_continuous(rng, n, t, hero=None):
    return np.stack([rng.uniform(0, 1, n), rng.uniform(-1, 1, n), rng.uniform(0, 1, n)], axis=1).astype(np.float32)


def test_c2_4096_lead_brake_autoreset_tables():
    """configs[1]: 4096 envs, lead_brake levels 1-3, continuous actions, trajectory tables on, auto-reset."""
    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.scenes import build_scripted_scene

    cls = load_map()
    scenes = [build_scripted_scene("lead_brake", i, level=1 + i % 3, cls_map=cls) for i in range(256)]
    n_auto, n_term, _ = run_scale_parity(scenes, 4096, steps=120, make_actions=_uniform_continuous,
                                      engine_kw=dict(action_mode=E.ACTION_CONTINUOUS),
                                      oracle_kw=dict(action_mode="continuous"), min_autoresets=64)
    assert n_term >= 64


@pytest.mark.parametrize("tables", [True, False])
def test_c3_8192_rdm_25_vehicles(tables):
    """configs[2] per-GPU shape: 8192 envs, rdm rt_hard_v1 (25 vehicles) from the shipped reference snapshots,
    discrete9 actions; with the open-loop trajectory tables and with live actor stepping (wide actor loops)."""
    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.config import ACTION_PROFILES
    from carlabev_env_b200.pool import load_shipped_pool

    scenes = load_shipped_pool("rdm_rt_hard_v1")

    def actions(rng, n, t, hero):
        return rng.choice(np.array([1, 1, 1, 3, 4, 0, 5, 6], dtype=np.int64), size=n)

    run_scale_parity(scenes, 8192, steps=120 if tables else 60, make_actions=actions,
                     engine_kw=dict(action_mode=E.ACTION_DISCRETE,
                                    discrete_table=ACTION_PROFILES["discrete9_v1"]["discrete_actions"],
                                    trajectory_steps=1024 if tables else 0),
                     oracle_kw=dict(action_mode="discrete"), min_autoresets=1)


def test_c4_8192_jaywalk_red_light_mix_autoreset():
    """configs[3] per-GPU shape: 8192 envs, 50/50 jaywalk (levels 1-4) / red_light_runner with traffic lights,
    continuous actions, auto-reset with mixed scene kinds; table -> live hand-over is crossed by using short tables."""
    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.pool import load_shipped_pool
    from carlabev_env_b200.scenes import build_scripted_scene

    cls = load_map()
    rl = load_shipped_pool("red_light_runner")
    scenes = []
    for i in range(64):
        scenes.append(build_scripted_scene("jaywalk", 7000 + i, level=1 + i % 4, cls_map=cls) if i % 2 == 0
                      else rl[(i // 2) % len(rl)])

    def actions(rng, n, t, hero):
        a = _uniform_continuous(rng, n, t)
        a[::2, 0] *= 0.25  # half of the envs crawl: the pedestrians' FSMs (incl. the StopReturn retreat) play out
        return a

    run_scale_parity(scenes, 8192, steps=120, make_actions=actions,
                     engine_kw=dict(action_mode=E.ACTION_CONTINUOUS, trajectory_steps=48),
                     oracle_kw=dict(action_mode="continuous"), min_autoresets=16)


@pytest.mark.parametrize("seed", [11, 12])
def test_engine_fuzz_with_pursuit_driving(seed):
    """tools/gpu_fuzz.py under pytest: random configurations, route-pursuit driving (long episodes, checkpoint and
    success endings), engine vs oracle."""
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "gpu_fuzz.py"), "2", str(seed), "220"], cwd=root,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "0 mismatching rounds" in r.stdout


@pytest.mark.parametrize("seed", [21])
def test_engine_fuzz_across_map_scales_and_observation_sizes(seed):
    """The same fuzzer drawing EnvConfig.size from {64, 128, 256} and the observation size from a list: k_render_any's
    block shortcut, its table / halving / copy / bilinear resizes and the scale factor of the sim kernels against the
    oracle (pinned on reference goldens at every scale and on cv2 for every resize branch)."""
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "gpu_fuzz.py"), "5", str(seed), "100", "1"], cwd=root,
                       capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "0 mismatching rounds" in r.stdout

"""Same-step auto-reset (AUTORESET_SAME_STEP, make_env(autoreset="same_step")) on the GPU.

The oracle is a twin engine in next_step mode with the same configuration, seed and pool.  The twin spends one extra
call per episode (its auto-reset call), so the two drift apart per env; actions are therefore a seeded function of
(env, episode, step within the episode), and every record is keyed by (env, episode, step).  For each key both engines
produced, the same-step engine must return the twin's reward, flags, cause, hero block and episode row bit for bit, and
the same window (a device-side 64-bit digest per env and call).  For each episode that ended, its final observation
must be the twin's window at the terminal call, its window after that call the twin's window after its auto-reset
call, and its new scene the twin's, all compared in full.  At the end each engine's statistics vector must be the sum
of the terminal episode rows it returned (so the two vectors agree up to the order of the atomics)."""
import numpy as np
import pytest

from test_gpu_action_repeat import _same_stats, _stats_from_rows
from test_gpu_lookahead_obs import TABLE
from test_gpu_snapshot import _engine, _rdm, _scripted

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]

M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def _hash(env, ep, k, seed):
    """splitmix64 of (seed, env, episode, step) per env: uint64 [N]."""
    with np.errstate(over="ignore"):
        z = (np.uint64(seed) * np.uint64(0x9E3779B97F4A7C15) + env.astype(np.uint64) * np.uint64(0xBF58476D1CE4E5B9)
             + ep.astype(np.uint64) * np.uint64(0x94D049BB133111EB) + k.astype(np.uint64) * np.uint64(0xD6E8FEB86659FD93))
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return (z ^ (z >> np.uint64(31))) & M64


def _acts(discrete, n_discrete, ep, k, seed, host=False):
    """The action row of every env at (its episode, its step within that episode)."""
    import torch

    z = _hash(np.arange(len(ep)), ep, k, seed)
    if discrete:
        a = (z % np.uint64(n_discrete)).astype(np.int64)
    else:
        # a steering side per episode: episodes end within tens of steps (off road, collisions)
        u = [((z >> np.uint64(s)) & np.uint64(0xFFFF)).astype(np.float64) / 65535.0 for s in (0, 16, 32)]
        side = np.where(_hash(np.arange(len(ep)), ep, np.zeros_like(k), seed) & np.uint64(1), 1.0, -1.0)
        a = np.stack([0.5 + 0.5 * u[0], side * (0.3 + 0.7 * u[1]), 0.1 * u[2]], axis=1).astype(np.float32)
    return a if host else torch.from_numpy(a).cuda()


class Digest:
    """64-bit digest per env of [N, ...] windows: the int32 words of each row times fixed random int64 weights, summed
    modulo 2^64 (integer sums do not depend on the reduction order)."""

    def __init__(self):
        self.coef = None

    def __call__(self, win):
        import torch

        w = win.reshape(win.shape[0], -1).contiguous()
        w = w.view(torch.int32).to(torch.int64) if w.dtype != torch.int64 else w
        if self.coef is None or self.coef.numel() < w.shape[1]:
            g = torch.Generator(device="cpu").manual_seed(7)
            self.coef = torch.randint(-(2**62), 2**62, (w.shape[1],), generator=g, dtype=torch.int64).cuda()
        return (w * self.coef[: w.shape[1]]).sum(1).cpu().numpy()


def _bits(x):
    return np.ascontiguousarray(x).view(np.int64) if isinstance(x, np.ndarray) else x.cpu().numpy().view(np.int64)


class Log:
    """Records of one engine keyed by (env, episode, step within the episode)."""

    def __init__(self):
        self.step = {}     # key -> (reward bits, term, trunc, cause, hero bits, digest or None)
        self.term = {}     # (env, ep) -> (terminal window, episode row)
        self.reset = {}    # (env, ep) -> (window after the reset, scene) of the episode ep starts
        self.rows = []


def _record(log, eng, envs, ep, k, digest, term_win=None):
    """One call's outputs of `envs` (host index array) into `log`; term_win: the terminal windows of this call's ended
    envs, [N, ...] (rows of ended envs valid)."""
    rew = eng.reward.cpu().numpy()
    te = eng.terminated.cpu().numpy().astype(bool)
    tr = eng.truncated.cpu().numpy().astype(bool)
    cause = eng.cause.cpu().numpy()
    hero = eng.hero.cpu().numpy()
    dig = digest(eng.obs())
    ended = te | tr
    for e in envs:
        key = (int(e), int(ep[e]), int(k[e]))
        log.step[key] = (_bits(rew[e:e + 1])[0], te[e], tr[e], cause[e], _bits(hero[e]).copy(),
                         None if ended[e] else dig[e])
        if ended[e]:
            row = eng.episode[e].clone()
            log.term[(int(e), int(ep[e]))] = ((term_win if term_win is not None else eng.obs())[e].clone(), row)
            log.rows.append(row.cpu().numpy())
    return ended


def _scene(eng, envs):
    import torch

    ids = torch.as_tensor(np.asarray(envs, dtype=np.int32)).cuda()
    return eng.snapshot(ids).header()[:, 0].cpu().numpy()


def run_same_step(a, calls, seed, digest):
    """Drive the same-step engine `a` for `calls` calls; returns its Log and the episodes each env finished."""
    from carlabev_env_b200 import engine as E

    N = a.N
    discrete = a.action_mode == E.ACTION_DISCRETE
    ep, k = np.zeros(N, np.int64), np.zeros(N, np.int64)
    log, allenv = Log(), np.arange(N)
    for _ in range(calls):
        a.step(_acts(discrete, a.cfg.n_discrete, ep, k, seed))
        ended = _record(log, a, allenv, ep, k, digest, term_win=a.final_obs)
        idx = np.flatnonzero(ended)
        if len(idx):
            obs = a.obs()
            for e, sc in zip(idx, _scene(a, idx)):
                log.reset[(int(e), int(ep[e]) + 1)] = (obs[e].clone(), int(sc))
        k += 1
        ep[ended] += 1
        k[ended] = 0
    return log, ep


def run_next_step(b, calls, seed, digest):
    """Drive the next_step twin `b`: an env whose last call ended spends this call on its auto-reset (action ignored),
    recorded as the reset of its next episode."""
    from carlabev_env_b200 import engine as E

    N = b.N
    discrete = b.action_mode == E.ACTION_DISCRETE
    ep, k = np.zeros(N, np.int64), np.zeros(N, np.int64)
    pending = np.zeros(N, bool)
    log = Log()
    for _ in range(calls):
        b.step(_acts(discrete, b.cfg.n_discrete, ep, k, seed))
        idx = np.flatnonzero(pending)
        if len(idx):
            assert not (b.terminated.cpu().numpy()[idx].any() or b.truncated.cpu().numpy()[idx].any())
            assert np.all(b.reward.cpu().numpy()[idx] == 0.0)
            obs = b.obs()
            for e, sc in zip(idx, _scene(b, idx)):
                log.reset[(int(e), int(ep[e]))] = (obs[e].clone(), int(sc))
        live = np.flatnonzero(~pending)
        ended = _record(log, b, live, ep, k, digest) & ~pending
        k[live] += 1
        pending[:] = ended
        ep[ended] += 1
        k[ended] = 0
    return log


def compare(la, lb):
    """Every key of `la` must be in `lb` with the same record; returns (steps, terminal episodes) compared."""
    import torch

    n_steps = 0
    for key, ra in la.step.items():
        rb = lb.step[key]
        assert ra[0] == rb[0], (key, "reward")
        assert ra[1:4] == rb[1:4], (key, "flags / cause", ra[1:4], rb[1:4])
        assert np.array_equal(ra[4], rb[4]), (key, "hero")
        assert (ra[5] is None) == (rb[5] is None) and (ra[5] is None or ra[5] == rb[5]), (key, "window digest")
        n_steps += 1
    for key, (wa, rowa) in la.term.items():
        wb, rowb = lb.term[key]
        assert torch.equal(wa, wb), (key, "final_obs against the twin's terminal window")
        assert torch.equal(rowa.view(torch.int64), rowb.view(torch.int64)), (key, "episode row")
    for key, (wa, sa) in la.reset.items():
        wb, sb = lb.reset[key]
        assert sa == sb, (key, "reset scene", sa, sb)
        assert torch.equal(wa, wb), (key, "reset window against the twin's auto-reset window")
    return n_steps, len(la.term)


def _pair(make, repeat=1):
    from carlabev_env_b200 import engine as E

    a, b = make(E.AUTORESET_SAME_STEP), make(E.AUTORESET_NEXT_STEP)
    for eng in (a, b):
        if repeat > 1:
            eng.set_action_repeat(repeat)
    return a, b


def _lead_brake():
    return _scripted(16, kinds=[("lead_brake", 1 + i % 3) for i in range(16)])


def _make_case(case):
    """(factory(autoreset) -> reset engine, action repeat, envs) of each configuration."""
    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.fovmask import corner_mask

    def reset(eng, n_scenes):
        eng.reset(np.arange(eng.N, dtype=np.int32) % n_scenes)
        return eng

    if case == "f32_lead_brake_carl":
        scenes = _lead_brake()
        return (lambda ar: reset(_engine(scenes, 48, autoreset=ar), len(scenes))), 1, 48
    if case == "u8_discrete_shaping_truncation_r4":
        scenes = _scripted(16)
        kw = dict(mask_dtype="uint8", action_mode=E.ACTION_DISCRETE, discrete_table=TABLE,
                  reward_mode=E.REWARD_SHAPING, reward_params={"max_actions": 9})
        return (lambda ar: reset(_engine(scenes, 48, autoreset=ar, **kw), len(scenes))), 4, 48
    if case == "gray64_fov_mask":
        scenes = _rdm(64)

        def make(ar):
            eng = _engine(scenes, 32, size=64, max_actors=16, obs_mode=E.OBS_GRAY, autoreset=ar)
            eng.upload_fov_mask(corner_mask(64, 0.5))
            return reset(eng, len(scenes))
        return make, 1, 32
    if case == "rgb_f1":
        scenes = _scripted(16)
        return (lambda ar: reset(_engine(scenes, 32, obs_mode=E.OBS_RGB, autoreset=ar), len(scenes))), 1, 32
    if case == "size256_live_actors":
        scenes = _rdm(256)
        kw = dict(size=256, max_actors=16, trajectory_steps=0)
        return (lambda ar: reset(_engine(scenes, 32, autoreset=ar, **kw), len(scenes))), 1, 32
    if case == "jaywalk_live_retreat":
        scenes = _scripted(16, kinds=[("jaywalk", 3 + i % 2) for i in range(16)])
        return (lambda ar: reset(_engine(scenes, 32, trajectory_steps=0, autoreset=ar), len(scenes))), 1, 32
    raise KeyError(case)


CASES = ["f32_lead_brake_carl", "u8_discrete_shaping_truncation_r4", "gray64_fov_mask", "rgb_f1",
         "size256_live_actors", "jaywalk_live_retreat"]


@pytest.mark.parametrize("case", CASES)
def test_same_step_equals_the_next_step_twin(case):
    make, repeat, n = _make_case(case)
    a, b = _pair(make, repeat)
    assert a.final_obs is not None and b.final_obs is None
    calls = 70
    seed = CASES.index(case)
    digest = Digest()
    la, eps = run_same_step(a, calls, seed, digest)
    # the twin needs one extra call per finished episode to reach every key of the same-step engine
    lb = run_next_step(b, calls + int(eps.max()) + 1, seed, digest)
    n_steps, n_term = compare(la, lb)
    assert n_steps == calls * n
    assert (eps >= 2).any(), ("want envs that end at least twice", eps)
    if case == "u8_discrete_shaping_truncation_r4":
        assert any(r[2] for r in la.step.values()), "want truncations"
    # statistics: each vector is the sum of the terminal rows it returned; the rows agree key by key (compare)
    from carlabev_env_b200 import engine as E

    for eng, log in ((a, la), (b, lb)):
        st = eng.read_stats().cpu().numpy()
        ref = _stats_from_rows(np.stack(log.rows) if log.rows else np.zeros((0, len(E.EPISODE_FIELDS))))
        st[-1] = ref[-1] = 0.0  # CBEV_S_STEPS counts calls
        _same_stats(st, ref, "statistics")
    a.close()
    b.close()


def test_launch_counts_per_call():
    """SAME_STEP calls issue 5 launches at repeat 1 and 4 above; next_step and disabled still 3 / 2 in one process."""
    import torch

    from carlabev_env_b200 import engine as E

    scenes = _scripted(8)
    rng = np.random.default_rng(0)
    for ar, want in ((E.AUTORESET_SAME_STEP, (5, 4)), (E.AUTORESET_NEXT_STEP, (3, 2)), (E.AUTORESET_DISABLED, (3, 2))):
        eng = _engine(scenes, 16, autoreset=ar)
        eng.reset(np.arange(16, dtype=np.int32) % 8)
        for rep, w in zip((1, 4), want):
            eng.set_action_repeat(rep)
            for _ in range(6):
                a = torch.from_numpy(np.stack([rng.uniform(0, 1, 16), rng.uniform(-1, 1, 16),
                                               np.zeros(16)], 1).astype(np.float32)).cuda()
                l0 = eng.launches
                if ar == E.AUTORESET_DISABLED and (eng.terminated | eng.truncated).any():
                    done = (eng.terminated | eng.truncated).bool()
                    eng.reset(np.zeros(16, dtype=np.int32), done)
                    l0 = eng.launches
                eng.step(a)
                assert eng.launches - l0 == w, (ar, rep)
        eng.close()


def _terminal_rows_of_twin(b, seed):
    """Step the next_step twin until some envs' last call ended; returns their ids (their snapshot rows are done)."""
    from carlabev_env_b200 import engine as E

    ep, k = np.zeros(b.N, np.int64), np.zeros(b.N, np.int64)
    for _ in range(200):
        b.step(_acts(b.action_mode == E.ACTION_DISCRETE, b.cfg.n_discrete, ep, k, seed))
        k += 1
        done = (b.terminated | b.truncated).cpu().numpy().astype(bool)
        if done.sum() >= 2:
            return np.flatnonzero(done)
    raise AssertionError("no terminal env")


def test_restored_terminal_row_auto_resets_as_next_step():
    """A terminal row restored into a SAME_STEP engine auto-resets at the next call exactly as under next_step: reward
    0, flags 0, the reset frame, the same scene and state; and both engines continue identically."""
    import torch

    from carlabev_env_b200 import engine as E

    scenes = _lead_brake()
    a, b = _pair(lambda ar: _engine(scenes, 32, autoreset=ar))
    for eng in (a, b):
        eng.reset(np.arange(32, dtype=np.int32) % 16)
    ended = _terminal_rows_of_twin(b, 3)
    snap = b.snapshot()
    assert (snap.header()[:, 2].cpu().numpy()[ended] == 1).all()
    a_info = a.snapshot().info
    a.restore(E.EnvSnapshot(snap._buf, a_info))  # same layout: B's rows go into A under A's own info
    b.restore(snap)
    assert torch.equal(a.obs(), b.obs())
    rng = np.random.default_rng(5)
    for s in range(12):
        acts = torch.from_numpy(np.stack([rng.uniform(0, 1, 32), rng.uniform(-1, 1, 32), np.zeros(32)],
                                         1).astype(np.float32)).cuda()
        a.step(acts)
        b.step(acts)
        if s == 0:
            assert (a.reward.cpu().numpy()[ended] == 0.0).all() and not a.terminated.cpu().numpy()[ended].any()
        for key in ("reward", "terminated", "truncated", "cause", "hero"):
            assert torch.equal(getattr(a, key), getattr(b, key)), (s, key)
        done = (b.terminated | b.truncated).bool()
        if done.any():  # from here on the two modes differ for these envs (b waits for its auto-reset call)
            assert torch.equal(a.final_obs[done], b.obs()[done]), s
            break
        assert torch.equal(a.obs(), b.obs()), s
        assert torch.equal(a.snapshot().data, b.snapshot().data), s
    a.close()
    b.close()


def test_lookahead_from_same_step_engine_equals_the_twin():
    """Plain, obs=True and row-rooted / leaf-row lookahead from a SAME_STEP engine equal the next_step twin's after the
    same snapshot rows (some terminal) are restored into both."""
    import torch

    from carlabev_env_b200 import engine as E

    scenes = _scripted(16)
    a, b = _pair(lambda ar: _engine(scenes, 32, autoreset=ar, action_mode=E.ACTION_DISCRETE, discrete_table=TABLE))
    for eng in (a, b):
        eng.reset(np.arange(32, dtype=np.int32) % 16)
    _terminal_rows_of_twin(b, 4)
    snap = b.snapshot()
    a.restore(E.EnvSnapshot(snap._buf, a.snapshot().info))
    b.restore(snap)
    rng = np.random.default_rng(9)
    acts = torch.from_numpy(rng.integers(0, len(TABLE), size=(12, 32))).cuda()
    for kw in (dict(), dict(obs=True), dict(obs=True, leaf=True)):
        la = a.lookahead(acts, rewards=True, hero=True, **kw)
        lb = b.lookahead(acts, rewards=True, hero=True, **kw)
        for key in ("ret", "steps", "terminated", "truncated", "cause", "reward", "hero", "obs"):
            x, y = getattr(la, key), getattr(lb, key)
            assert (x is None) == (y is None) and (x is None or torch.equal(x, y)), (kw, key)
        if kw.get("leaf"):
            assert torch.equal(la.leaf.data, lb.leaf.data)
            ra = a.lookahead(acts, obs=True, source=la.leaf, leaf=True)
            rb = b.lookahead(acts, obs=True, source=lb.leaf, leaf=True)
            for key in ("ret", "steps", "obs"):
                assert torch.equal(getattr(ra, key), getattr(rb, key)), ("rows", key)
            assert torch.equal(ra.leaf.data, rb.leaf.data)
    a.close()
    b.close()


# ---- make_env ------------------------------------------------------------------------------------------------------
def _vec_twin(kw_env, kw_make, calls=50, seed=0):
    """make_env(autoreset="same_step") against make_env(autoreset="next_step") with keyed actions: per (env, episode,
    step) the rewards and flags, per finished episode the final observation (against the twin's observation at its
    terminal call) and final_info's episode_info / episode (against the twin's top-level terminal keys)."""
    import torch

    from carlabev_env_b200.config import EnvConfig, RunConfig
    from carlabev_env_b200.vector_env import make_env

    scenes = _scripted(16)
    cfg = RunConfig(env=EnvConfig(**kw_env), num_envs=kw_make.pop("num_envs", 24))
    envs = {m: make_env(cfg, scenes=scenes, autoreset=m, ring_budget_bytes=32 << 20, **kw_make)
            for m in ("same_step", "next_step")}
    for v in envs.values():
        v.reset(options={"scene": "pool"})
    sa, nb = envs["same_step"], envs["next_step"]
    assert sa.metadata["autoreset_mode"] in ("SameStep",) or "SAME_STEP" in str(sa.metadata["autoreset_mode"])
    N = sa.num_envs
    discrete = kw_env.get("action_mode", "discrete") == "discrete"
    n_disc = sa.single_action_space.n if discrete else 0
    to_np = kw_make.get("to_numpy", False)
    host = kw_make.get("host_infos", True)

    def arr(x):
        return x if isinstance(x, np.ndarray) else x.cpu().numpy()

    recs = {"same_step": ({}, {}), "next_step": ({}, {})}
    ended_twice = 0
    for mode, v in envs.items():
        ep, k = np.zeros(N, np.int64), np.zeros(N, np.int64)
        pending = np.zeros(N, bool)
        steps, terms = recs[mode]
        for _ in range(calls if mode == "same_step" else calls + 40):
            obs, rew, term, trunc, infos = v.step(_acts(discrete, n_disc, ep, k, seed, host=True))
            assert "hero" in infos and "cause" in infos
            rew, term, trunc = arr(rew), arr(term).astype(bool), arr(trunc).astype(bool)
            done = (term | trunc) & ~pending
            for e in np.flatnonzero(~pending):
                steps[(e, ep[e], k[e])] = (rew[e], term[e], trunc[e])
            if mode == "same_step":
                if not host:
                    assert torch.equal(infos["_final_obs"], torch.from_numpy(done).cuda())
                    fin = infos["final_obs"]
                    info = None
                elif done.any():
                    assert "episode_info" not in infos and "episode" not in infos
                    assert np.array_equal(infos["_final_obs"], done) and np.array_equal(infos["_final_info"], done)
                    fin = infos["final_obs"]
                    if to_np:
                        assert fin.dtype == object and all(fin[e] is None for e in np.flatnonzero(~done))
                    info = infos["final_info"]
                else:
                    assert "final_obs" not in infos and "final_info" not in infos
                for e in np.flatnonzero(done):
                    o = fin[e] if to_np else fin[e].clone()
                    terms[(e, ep[e])] = (o, None if info is None else
                                         (info["episode_info"]["return"][e], info["episode"]["l"][e]))
                k += 1
                ep[done] += 1
                k[done] = 0
            else:
                for e in np.flatnonzero(done):
                    o = obs[e] if to_np else obs[e].clone()
                    terms[(e, ep[e])] = (o, (infos["episode_info"]["return"][e], infos["episode"]["l"][e])
                                         if "episode_info" in infos else None)
                live = ~pending
                k[live] += 1
                pending = done
                ep[done] += 1
                k[done] = 0
        if mode == "same_step":
            ended_twice = int((ep >= 2).sum())
    (sa_steps, sa_terms), (nb_steps, nb_terms) = recs["same_step"], recs["next_step"]
    for key, r in sa_steps.items():
        assert nb_steps[key][0].tobytes() == r[0].tobytes() and nb_steps[key][1:] == r[1:], key
    assert sa_terms, "no episode ended"
    for key, (o, inf) in sa_terms.items():
        ob, infb = nb_terms[key]
        if to_np:
            assert np.array_equal(o, ob), key
        else:
            assert torch.equal(o, ob), key
        if inf is not None:
            assert inf[0] == infb[0] and inf[1] == infb[1], (key, inf, infb)
    assert ended_twice > 0
    for v in envs.values():
        v.close()


@pytest.mark.parametrize("variant", ["stack", "vehicle_temporal", "vehicle_weighted", "to_numpy", "async",
                                     "repeat4", "shard"])
def test_make_env_same_step_against_next_step(variant):
    kw_env = dict(action_mode="continuous")
    kw_make = {}
    if variant in ("vehicle_temporal", "vehicle_weighted"):
        kw_env["temporal_fusion_mode"] = variant
    elif variant == "to_numpy":
        kw_make["to_numpy"] = True
    elif variant == "async":
        kw_make["host_infos"] = False
    elif variant == "repeat4":
        kw_make["action_repeat"] = 4
    elif variant == "shard":
        kw_make.update(shard=(1, 2), num_envs=40)
    _vec_twin(kw_env, kw_make)

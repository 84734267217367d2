"""Lookahead with rendered leaf observations (Engine.lookahead(obs=True) / cbev_lookahead_obs, cbev_fuse_windows) on
the GPU.

The reference is the clone-and-step recipe of test_gpu_lookahead.py: the roots' snapshot rows are restored as clones
into the envs of the same engine (auto-reset disabled) and stepped with the branches' actions; `Engine.obs()` (or
`Engine.fuse(mode)`) of each clone right after its branch's last step must equal the leaf window byte for byte.  A
branch with steps = 0 shows its root's current window (terminal root) or zeros (a device root outside [0, N)).  The
rest of the result must be bit-identical to the same call without observations, and the live engine must be left
as it was."""
import numpy as np
import pytest

from test_gpu_lookahead import _live_state, _plan_actions, _same_state, _warm
from test_gpu_snapshot import _actions, _rdm, _scripted

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]

RESULT_FIELDS = ("ret", "reward", "steps", "terminated", "truncated", "cause", "hero")
TABLE = np.asarray([[0, 0, 0], [1, 0, 0], [0.5, -1, 0], [0.5, 1, 0], [0, 0, 1], [1, -0.5, 0], [1, 0.5, 0]],
                   dtype=np.float32)


def _engine(scenes, n, size=128, **kw):
    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.pool import pack_pool
    from golden_util import load_map

    args = dict(mask_mode="6-class", frame_stack=4, ring_slots=7, action_mode=E.ACTION_CONTINUOUS,
                autoreset=E.AUTORESET_DISABLED, max_actors=4, seed=3, size=size)
    args.update(kw)
    if args.get("obs_mode") == E.OBS_RGB:
        args["ring_slots"] = None
    eng = E.Engine(n, **args)
    eng.upload_map(load_map(size))
    eng.upload_pool(pack_pool(scenes))
    return eng


def _reference(eng, snap, roots, acts, steps, root_obs, fuse=None):
    """Leaf window (or its fusion) of every branch from clones stepped in the live engine, in chunks of at most N
    branches; only branches with steps > 0 are stepped.  Restores the whole snapshot afterwards."""
    import torch

    N, B = eng.N, len(roots)
    out = torch.zeros((B,) + tuple(root_obs.shape[1:]), dtype=root_obs.dtype, device=root_obs.device)
    valid = (roots >= 0) & (roots < N)
    for b in np.flatnonzero((steps == 0) & valid):
        out[b] = root_obs[roots[b]]
    idx = np.flatnonzero(steps > 0)
    for c0 in range(0, len(idx), N):
        chunk = idx[c0:c0 + N]
        k = len(chunk)
        eng.restore(snap, env_ids=np.arange(k), rows=roots[chunk])
        sel = torch.from_numpy(chunk).to(acts.device)
        for t in range(int(steps[chunk].max())):
            a = torch.zeros((N,) + tuple(acts.shape[2:]), dtype=acts.dtype, device=acts.device)
            a[:k] = acts[t].index_select(0, sel)
            eng.step(a)
            o = eng.obs() if fuse is None else eng.fuse(fuse)
            for i in np.flatnonzero(steps[chunk] == t + 1):
                out[chunk[i]] = o[i]
    eng.restore(snap)
    return out


def _check(eng, rng, roots, H, fuse=None, acts=None):
    """Lookahead with observations from `roots` (host array, or int32 CUDA tensor) against the call without them and
    against the stepping reference; returns the result."""
    import torch

    roots_np = roots.cpu().numpy() if isinstance(roots, torch.Tensor) else np.asarray(roots)
    B = len(roots_np)
    if acts is None:
        acts = _plan_actions(eng, rng, H, B)
    snap = eng.snapshot()
    root_obs = (eng.obs() if fuse is None else eng.fuse(fuse)).clone()
    plain = eng.lookahead(acts, env_ids=roots, rewards=True, hero=True)
    plain = {k: getattr(plain, k).clone() for k in RESULT_FIELDS}
    la = eng.lookahead(acts, env_ids=roots, rewards=True, hero=True, obs=True, fuse=fuse)
    for k in RESULT_FIELDS:
        assert torch.equal(getattr(la, k), plain[k]), k
    steps = la.steps.cpu().numpy()
    shape = (B,) + tuple(root_obs.shape[1:])
    assert tuple(la.obs.shape) == shape and la.obs.dtype == root_obs.dtype, (la.obs.shape, la.obs.dtype)
    ref = _reference(eng, snap, roots_np, acts, steps, root_obs, fuse)
    bad = [b for b in range(B) if not torch.equal(la.obs[b], ref[b])]
    assert not bad, (len(bad), bad[:8], steps[bad[:8]])
    return la


CASES = ["f32", "u8", "binary", "2-class", "4-class", "5-class", "7-class", "gray75", "rgb", "size64", "size256",
         "obs84", "fov_masked", "dbg1", "dbg256", "dbg512", "discrete", "traj0", "traj8", "jaywalk_stop_return",
         "red_light_runner"]


@pytest.mark.parametrize("case", CASES)
def test_leaf_windows_equal_stepping(case):
    from carlabev_env_b200 import engine as E

    n, size, kw, scenes, warm, H, dbg = 32, 128, {}, None, 12, 24, 0
    if case == "u8":
        kw["mask_dtype"] = "uint8"
    elif case in ("binary", "4-class", "7-class"):
        kw["mask_mode"] = case
    elif case in ("2-class", "5-class"):
        kw.update(mask_mode=case, mask_dtype="uint8")
    elif case == "gray75":
        kw.update(obs_mode=E.OBS_GRAY, anchor=(0.5, 0.75))
    elif case == "rgb":
        kw["obs_mode"] = E.OBS_RGB
    elif case in ("size64", "size256", "dbg512"):
        size = 64 if case == "size64" else 256
        scenes, kw["max_actors"] = _rdm(size), 16
        dbg = 512 if case == "dbg512" else 0  # 256 -> 96 takes k_render_any's 8:3 shortcut unless flag 512
    elif case == "obs84":
        kw["obs_size"] = (84, 84)
    elif case in ("dbg1", "dbg256"):
        dbg = int(case[3:])
    elif case == "discrete":
        kw.update(action_mode=E.ACTION_DISCRETE, discrete_table=TABLE)
    elif case == "traj0":
        kw["trajectory_steps"] = 0
    elif case == "traj8":
        kw["trajectory_steps"] = 8
        warm = 3  # the table -> live hand-over (episode step 8) happens inside the horizon
    elif case == "jaywalk_stop_return":
        scenes = _scripted(16, kinds=[("jaywalk", 3 + i % 2) for i in range(16)])
        kw["trajectory_steps"] = 0
        warm, H = 8, 64  # walkers yield, then start their retreat inside the horizon
    elif case == "red_light_runner":
        from carlabev_env_b200.scenes import build_pool

        scenes = build_pool([dict(scene="red_light_runner", scene_seed=i) for i in range(8)], pad=182)
        kw["max_actors"] = max(len(s["act_kind"]) for s in scenes)
    if scenes is None:
        scenes = _scripted(16)
    eng = _engine(scenes, n, size=size, **kw)
    if case == "fov_masked":
        from carlabev_env_b200.fovmask import corner_mask

        eng.upload_fov_mask(corner_mask(128, 0.5))
    if dbg:
        eng.set_debug_flags(dbg)
    eng.reset(np.arange(n, dtype=np.int32) % len(scenes))
    rng = np.random.default_rng(CASES.index(case))
    _warm(eng, rng, warm)
    _check(eng, rng, np.arange(n), H)
    la = _check(eng, rng, rng.integers(0, n, size=3 * n // 2), H)  # repeated roots, B > N
    if case == "f32":
        s = la.steps.cpu().numpy()
        assert ((s > 0) & (s < H)).any(), "want branches that end inside the horizon"
    eng.close()


def test_window_composition():
    """H < F, branches that end at steps 1..F-1 (shaping's max_actions truncation), roots whose window holds reset
    frames, roots whose window lies in the ring's mirror zone, terminal roots, out-of-range device roots."""
    import torch

    from carlabev_env_b200 import engine as E

    n, F, L = 16, 4, 7
    scenes = _scripted(16)
    eng = _engine(scenes, n, action_mode=E.ACTION_DISCRETE, discrete_table=TABLE, reward_mode=E.REWARD_SHAPING,
                  reward_params={"max_actions": 30})
    eng.reset(np.arange(n, dtype=np.int32))
    rng = np.random.default_rng(2)
    for H in (1, 2, 3, 5):  # the window still holds the reset frames
        _check(eng, rng, rng.integers(0, n, size=24), H)
    heads, ended = set(), set()
    for k in range(1, 30):
        _warm(eng, rng, 1)
        heads.add(eng.head)
        H = 8 if k >= 26 else 1 + k % 3
        la = _check(eng, rng, rng.integers(0, n, size=24), H)
        s = la.steps.cpu().numpy()
        ended |= set(s[(la.truncated | la.terminated).cpu().numpy().astype(bool)].tolist())
    assert heads == set(range(F - 1, L)), heads  # every head position, the mirror zone (head >= L - F + 1) included
    assert {1, 2, 3} <= ended, ended
    _warm(eng, rng, 1)  # step 30: every env truncated, waiting for a reset
    la = _check(eng, rng, rng.integers(0, n, size=24), 4)
    assert not la.steps.any()
    eng.reset(np.arange(n, dtype=np.int32))
    _warm(eng, rng, 5)
    bad = torch.tensor([-1, n, 0, 10 ** 6, 3], dtype=torch.int32, device=eng.device)
    la = _check(eng, rng, bad, 6)
    assert la.steps.cpu().tolist()[:2] == [0, 0] and la.steps[3].item() == 0
    assert not la.obs[[0, 1, 3]].any()
    eng.close()


@pytest.mark.parametrize("dtype", ["float32", "uint8"])
@pytest.mark.parametrize("mode", ["vehicle_temporal", "vehicle_weighted"])
def test_fused_leaf_windows_equal_stepping(mode, dtype):
    n = 32
    eng = _engine(_scripted(16), n, mask_dtype=dtype)
    eng.reset(np.arange(n, dtype=np.int32) % 16)
    rng = np.random.default_rng(11)
    _warm(eng, rng, 10)
    la = _check(eng, rng, rng.integers(0, n, size=48), 20, fuse=mode)
    assert la.window is not None and la.window is not la.obs
    assert tuple(la.window.shape) == (48,) + tuple(eng.obs().shape[1:])
    eng.close()


def test_live_engine_is_untouched():
    """Against a twin engine that never looks ahead: ring, snapshot rows, statistics and last outputs identical after
    an obs lookahead with B > N and repeated roots, and every output identical over the next 16 steps."""
    from carlabev_env_b200 import engine as E

    scenes = _scripted(16)
    n = 64
    engs = [_engine(scenes, n, autoreset=E.AUTORESET_NEXT_STEP) for _ in range(2)]
    rng = np.random.default_rng(17)
    for e in engs:
        e.reset(np.arange(n, dtype=np.int32) % len(scenes))
    for _ in range(25):
        a = _actions(rng, n)
        for e in engs:
            e.step(a)
    before = _live_state(engs[0])
    launches = engs[0].launches
    acts = _plan_actions(engs[0], rng, 32, 4 * n)
    la = engs[0].lookahead(acts, env_ids=rng.integers(0, n, size=4 * n), rewards=True, hero=True, obs=True)
    assert engs[0].launches == launches + 3
    assert (la.terminated.cpu().numpy() & (la.steps.cpu().numpy() > 0)).any(), "no branch ended an episode"
    la = engs[0].lookahead(acts, env_ids=rng.integers(0, n, size=4 * n), obs=True, fuse="vehicle_temporal")
    assert engs[0].launches == launches + 7
    _same_state(before, _live_state(engs[0]), "after lookahead")
    _same_state(_live_state(engs[1]), _live_state(engs[0]), "twin", twin=True)
    for t in range(16):
        a = _actions(rng, n)
        for e in engs:
            e.step(a)
        _same_state(_live_state(engs[1]), _live_state(engs[0]), f"{t + 1} steps later", twin=True)
    for e in engs:
        e.close()


def _more_lights(a, b):
    """Scene a with the traffic lights of scene b added (a larger max_tl, so a longer draw list per env)."""
    s = dict(a)
    s["tl_rect"] = np.concatenate([np.asarray(a["tl_rect"]).reshape(-1, 4), np.asarray(b["tl_rect"]).reshape(-1, 4)])
    s["tl_color"] = np.concatenate([np.asarray(a["tl_color"]), np.asarray(b["tl_color"])])
    return s


def test_growth_and_out_reuse():
    """The branch render state grows with B and when an append-only pool extension raises max_rects; `out=` reuse
    gives the bytes of a fresh call."""
    import torch

    from carlabev_env_b200.pool import pack_pool
    from carlabev_env_b200.scenes import build_pool

    scenes = build_pool([dict(scene="red_light_runner", scene_seed=i) for i in range(8)], pad=182)
    n = 24
    eng = _engine(scenes, n, max_actors=max(len(s["act_kind"]) for s in scenes))
    eng.reset(np.arange(n, dtype=np.int32) % len(scenes))
    rng = np.random.default_rng(4)
    _warm(eng, rng, 6)
    _check(eng, rng, rng.integers(0, n, size=8), 12)
    _check(eng, rng, rng.integers(0, n, size=3 * n), 12)  # B grows
    grown = scenes + [_more_lights(scenes[i], scenes[i + 1]) for i in range(0, 8, 2)]
    assert max(len(s["tl_color"]) for s in grown) > max(len(s["tl_color"]) for s in scenes)
    eng.upload_pool(pack_pool(grown))  # append-only: max_rects grows with max_tl
    eng.reset(np.arange(n, dtype=np.int32) % len(grown))
    _warm(eng, rng, 6)
    _check(eng, rng, rng.integers(0, n, size=3 * n), 12)  # same B, longer draw lists
    _check(eng, rng, rng.integers(0, n, size=4 * n), 12, fuse="vehicle_weighted")
    acts = _plan_actions(eng, rng, 9, 40)
    roots = rng.integers(0, n, size=40)
    r1 = eng.lookahead(_plan_actions(eng, rng, 9, 40), env_ids=roots, obs=True, fuse="vehicle_temporal")
    earlier = r1.window.clone()
    r3 = eng.lookahead(acts, env_ids=roots, obs=True, fuse="vehicle_temporal")
    r2 = eng.lookahead(acts, env_ids=roots, obs=True, fuse="vehicle_temporal", out=r1)
    assert r2 is r1 and not torch.equal(earlier, r3.window)
    for k in ("obs", "window", "ret", "steps"):
        assert torch.equal(getattr(r2, k), getattr(r3, k)), k
    eng.close()


def test_value_errors():
    from carlabev_env_b200 import engine as E

    eng = _engine(_scripted(8), 8)
    eng.reset(np.arange(8, dtype=np.int32))
    rng = np.random.default_rng(0)
    acts = _plan_actions(eng, rng, 4, 8)
    with pytest.raises(ValueError, match="needs obs=True"):
        eng.lookahead(acts, fuse="vehicle_temporal")
    with pytest.raises(ValueError, match="fuse must be one of"):
        eng.lookahead(acts, obs=True, fuse="vehicle")
    r = eng.lookahead(acts)
    with pytest.raises(ValueError, match="leaf-window buffer"):
        eng.lookahead(acts, obs=True, out=r)
    r = eng.lookahead(acts, obs=True)
    with pytest.raises(ValueError, match="buffer for fuse"):
        eng.lookahead(acts, obs=True, fuse="vehicle_weighted", out=r)
    r = eng.lookahead(acts, obs=True, fuse="vehicle_temporal")
    with pytest.raises(ValueError, match="buffer for fuse"):
        eng.lookahead(acts, obs=True, fuse="vehicle_weighted", out=r)
    eng.close()
    eng = _engine(_scripted(8), 8, obs_mode=E.OBS_GRAY)
    eng.reset(np.arange(8, dtype=np.int32))
    with pytest.raises(ValueError, match="bev_semantic"):
        eng.lookahead(acts, obs=True, fuse="vehicle_temporal")
    eng.close()


@pytest.mark.parametrize("workload", ["c2", "c3"])
def test_scale(workload):
    """4096 branches on the c2 workload (lead_brake pool, continuous, float32 masks), every one against stepping; 8192
    on a c3-style pool (25-vehicle rt_hard_v1 scenes stepped live: the 32-lane path, discrete, uint8 masks), a seeded
    sample of 256 against stepping."""
    import torch

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.vector_env import load_town01_map

    if workload == "c2":
        n = 4096
        eng = E.Engine(n, ring_slots=7, action_mode=E.ACTION_CONTINUOUS, autoreset=E.AUTORESET_DISABLED, max_actors=4,
                       seed=0)
        eng.upload_map(load_town01_map(128))
        k = 1024
        eng.generate_scripted_pool(["lead_brake"] * k, [1 + i % 3 for i in range(k)], list(range(k)))
    else:
        from carlabev_env_b200.pool import pack_pool
        from carlabev_env_b200.reset import RandomNavigationReset, build_reset_options
        from carlabev_env_b200.scenes import build_pool

        n, k = 8192, 32
        scenes = build_pool([build_reset_options(RandomNavigationReset(difficulty_id="rt_hard_v1", scene_seed=i))
                             for i in range(k)], pad=182)
        table = np.asarray([[0, 0, 0], [1, 0, 0], [0.5, -1, 0], [0.5, 1, 0], [0, 0, 1]], dtype=np.float32)
        eng = E.Engine(n, ring_slots=7, action_mode=E.ACTION_DISCRETE, discrete_table=table,
                       autoreset=E.AUTORESET_DISABLED, max_actors=25, trajectory_steps=0, seed=0, mask_dtype="uint8")
        eng.upload_map(load_town01_map(128))
        eng.upload_pool(pack_pool(scenes))
    eng.reset(np.arange(n, dtype=np.int32) % k)
    rng = np.random.default_rng(1)
    _warm(eng, rng, 10)
    if workload == "c2":
        _check(eng, rng, np.arange(n), 8)
    else:
        roots = np.arange(n)
        acts = _plan_actions(eng, rng, 8, n)
        snap = eng.snapshot()
        root_obs = eng.obs().clone()
        la = eng.lookahead(acts, env_ids=roots, obs=True)
        sample = np.sort(np.random.default_rng(8).choice(n, size=256, replace=False))
        sel = torch.from_numpy(sample).cuda()
        steps = la.steps.cpu().numpy()[sample]
        ref = _reference(eng, snap, roots[sample], acts.index_select(1, sel).contiguous(), steps, root_obs)
        assert torch.equal(la.obs.index_select(0, sel), ref)
    eng.close()

"""Lookahead from snapshot rows and leaf snapshot rows (Engine.lookahead(source=, rows=, leaf=True) /
cbev_lookahead_ex) on the GPU.

The reference for a leaf row is the clone-and-step recipe: the root row is restored into an env of the same engine
(auto-reset disabled), stepped with the branch's actions, and snapshotted right after the branch's own last step;
`la.leaf` row b must equal that snapshot byte for byte, padding included.  A call from rows must reproduce every output
of the call from the live envs the rows were taken from, a leaf row must continue bit-identically both as the root of
the next call and restored into a live env, and the live engine must be left as it was."""
import ctypes as C

import numpy as np
import pytest

from test_gpu_lookahead import _live_state, _plan_actions, _ret_numpy, _same_state, _warm
from test_gpu_lookahead_obs import TABLE, _engine
from test_gpu_snapshot import _rdm, _scripted, _two_walkers

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]

FIELDS = ("ret", "reward", "steps", "terminated", "truncated", "cause", "hero", "obs")
SENTINEL = 0xA5


def _results(la):
    return {k: getattr(la, k).clone() for k in FIELDS if getattr(la, k) is not None}


def _same_results(a, b, what):
    for k in a:
        assert np.array_equal(a[k].cpu().numpy(), b[k].cpu().numpy()), (what, k)


def _leaf_reference(eng, src, rows, acts, steps, valid):
    """Snapshot row of every valid branch's leaf from clones of its root row stepped in the live engine (chunks of at
    most N branches), SENTINEL bytes for the others.  Restores the live state afterwards."""
    import torch

    live = eng.snapshot()
    N, B = eng.N, len(rows)
    ref = torch.full((B, eng.snapshot_row_bytes), SENTINEL, dtype=torch.uint8, device=eng.device)
    idx = np.flatnonzero(valid)
    for c0 in range(0, len(idx), N):
        chunk = idx[c0:c0 + N]
        k = len(chunk)
        eng.restore(src, env_ids=np.arange(k), rows=rows[chunk])
        sel = torch.from_numpy(chunk).to(acts.device)
        for t in range(int(steps[chunk].max()) + 1):
            at = np.flatnonzero(steps[chunk] == t)
            if len(at):
                ref[torch.from_numpy(chunk[at]).to(eng.device)] = eng.snapshot(env_ids=at).data
            if t == int(steps[chunk].max()):
                break
            a = torch.zeros((N,) + tuple(acts.shape[2:]), dtype=acts.dtype, device=acts.device)
            a[:k] = acts[t].index_select(0, sel)
            eng.step(a)
    eng.restore(live)
    return ref


def _check_leaf(eng, rng, roots, H, acts=None):
    """Live roots with leaf rows (and windows) against the plain calls and the stepping reference.  Returns
    (result, actions, snapshot of the roots' engine before the call)."""
    import torch

    B = len(roots)
    if acts is None:
        acts = _plan_actions(eng, rng, H, B)
    snap = eng.snapshot()
    plain = _results(eng.lookahead(acts, env_ids=roots, rewards=True, hero=True, obs=True))
    la = eng.lookahead(acts, env_ids=roots, rewards=True, hero=True, obs=True, leaf=True)
    _same_results(plain, _results(la), "leaf=True changes the results")
    assert la.leaf.n_rows == B and la.leaf.row_bytes == eng.snapshot_row_bytes
    assert la.leaf.info.retreat_slots == snap.info.retreat_slots and la.leaf.info.pool_epoch == snap.info.pool_epoch
    # without obs the windows go to engine scratch: same rows
    la2 = eng.lookahead(acts, env_ids=roots, leaf=True)
    assert torch.equal(la2.leaf.data, la.leaf.data)
    steps = la.steps.cpu().numpy()
    valid = (np.asarray(roots) >= 0) & (np.asarray(roots) < eng.N)
    ref = _leaf_reference(eng, snap, np.asarray(roots), acts, steps, valid)
    bad = [b for b in range(B) if not torch.equal(la.leaf.data[b], ref[b])]
    assert not bad, (len(bad), bad[:8], steps[bad[:8]])
    return la, acts, snap


def _check_rows_equal_live(eng, rng, snap, roots, acts, live_res, live_leaf):
    """After the live batch moved on: the call from the rows of `snap` reproduces the call from the live envs."""
    import torch

    _warm(eng, rng, 3)
    before = _live_state(eng)
    la = eng.lookahead(acts, source=snap, rows=roots, rewards=True, hero=True, obs=True, leaf=True)
    _same_results(live_res, _results(la), "rows as roots")
    assert torch.equal(la.leaf.data, live_leaf)
    plain = eng.lookahead(acts, source=snap, rows=roots, rewards=True, hero=True)  # the observation-free kernel
    _same_results({k: v for k, v in live_res.items() if k != "obs"}, _results(plain), "rows as roots, no obs")
    _same_state(before, _live_state(eng), "rows as roots")


CASES = ["f32", "u8", "gray", "rgb", "size64", "size256", "obs84", "discrete", "shaping_truncation", "traj0", "traj8",
         "jaywalk_stop_return", "red_light_runner", "c3_wide"]


@pytest.mark.parametrize("case", CASES)
def test_leaf_rows_equal_snapshots_of_stepped_clones(case):
    from carlabev_env_b200 import engine as E

    n, size, kw, scenes, warm, H = 32, 128, {}, None, 12, 24
    if case == "u8":
        kw["mask_dtype"] = "uint8"
    elif case == "gray":
        kw["obs_mode"] = E.OBS_GRAY
    elif case == "rgb":
        kw["obs_mode"] = E.OBS_RGB
    elif case in ("size64", "size256"):
        size = 64 if case == "size64" else 256
        scenes, kw["max_actors"] = _rdm(size), 16
    elif case == "obs84":
        kw["obs_size"] = (84, 84)
    elif case == "discrete":
        kw.update(action_mode=E.ACTION_DISCRETE, discrete_table=TABLE)
    elif case == "shaping_truncation":
        kw.update(action_mode=E.ACTION_DISCRETE, discrete_table=TABLE, reward_mode=E.REWARD_SHAPING,
                  reward_params={"max_actions": 20})
        warm = 4  # every branch truncates inside the horizon
    elif case == "traj0":
        kw["trajectory_steps"] = 0
    elif case == "traj8":
        kw["trajectory_steps"] = 8
        warm = 3  # the table -> live hand-over happens inside the horizon
    elif case == "jaywalk_stop_return":
        scenes = _scripted(16, kinds=[("jaywalk", 3 + i % 2) for i in range(16)])
        kw["trajectory_steps"] = 0
        warm, H = 8, 64
    elif case == "red_light_runner":
        from carlabev_env_b200.scenes import build_pool

        scenes = build_pool([dict(scene="red_light_runner", scene_seed=i) for i in range(8)], pad=182)
        kw["max_actors"] = max(len(s["act_kind"]) for s in scenes)
    elif case == "c3_wide":
        from carlabev_env_b200.reset import RandomNavigationReset, build_reset_options
        from carlabev_env_b200.scenes import build_pool

        scenes = build_pool([build_reset_options(RandomNavigationReset(difficulty_id="rt_hard_v1", scene_seed=i))
                             for i in range(8)], pad=182)
        kw.update(max_actors=25, trajectory_steps=0, mask_dtype="uint8")  # live-stepped 25 vehicles: G = 32
    if scenes is None:
        scenes = _scripted(16)
    eng = _engine(scenes, n, size=size, **kw)
    eng.reset(np.arange(n, dtype=np.int32) % len(scenes))
    rng = np.random.default_rng(CASES.index(case))
    _warm(eng, rng, warm)
    roots = rng.integers(0, n, size=3 * n // 2)  # repeated roots, B > N
    la, acts, snap = _check_leaf(eng, rng, roots, H)
    s = la.steps.cpu().numpy()
    if case in ("f32", "shaping_truncation"):
        assert ((s > 0) & (s < H)).any(), "want branches that end inside the horizon"
    _check_rows_equal_live(eng, rng, snap, roots, acts, _results(la), la.leaf.data.clone())
    eng.close()


def test_chaining_equals_one_call():
    """H1 steps, then H2 more from la.leaf, against one H1 + H2 call: per-step rewards, flags, cause, hero, leaf
    window and leaf rows; ret recomputed in NumPy from the concatenated rewards (summation order differs)."""
    import torch

    from carlabev_env_b200 import engine as E

    n = 32
    eng = _engine(_scripted(16), n, action_mode=E.ACTION_DISCRETE, discrete_table=TABLE,
                  reward_mode=E.REWARD_SHAPING, reward_params={"max_actions": 26})
    eng.reset(np.arange(n, dtype=np.int32) % 16)
    rng = np.random.default_rng(5)
    _warm(eng, rng, 6)
    for H1, H2 in ((1, 3), (3, 2), (5, 16)):  # H < F on both sides; truncation inside either part
        roots = rng.integers(0, n, size=48)
        acts = _plan_actions(eng, rng, H1 + H2, 48)
        full = eng.lookahead(acts, env_ids=roots, rewards=True, hero=True, obs=True, leaf=True)
        a = eng.lookahead(acts[:H1].contiguous(), env_ids=roots, rewards=True, hero=True, obs=True, leaf=True)
        b = eng.lookahead(acts[H1:].contiguous(), source=a.leaf, rewards=True, hero=True, obs=True, leaf=True)
        s1, s2 = a.steps.cpu().numpy(), b.steps.cpu().numpy()
        assert np.array_equal(full.steps.cpu().numpy(), s1 + s2)
        assert not s2[s1 < H1].any() and not (a.terminated | a.truncated).cpu().numpy()[s2 > 0].any()
        rew = torch.cat([a.reward, b.reward])
        assert torch.equal(full.reward, rew)
        assert np.array_equal(full.ret.cpu().numpy(), _ret_numpy(rew.cpu().numpy(), s1 + s2, 1.0))
        cont = torch.from_numpy(s2 > 0).to(eng.device)
        for k in ("terminated", "truncated", "cause"):
            assert torch.equal(getattr(full, k), torch.where(cont, getattr(b, k), getattr(a, k))), k
        assert torch.equal(full.hero, torch.where(cont[:, None], b.hero, a.hero))
        assert torch.equal(full.obs, b.obs)
        assert torch.equal(full.leaf.data, b.leaf.data)
    eng.close()


def test_leaf_row_restored_and_stepped_continues_the_clone():
    import torch

    n, H, K = 24, 10, 12
    eng = _engine(_scripted(16), n)
    eng.reset(np.arange(n, dtype=np.int32) % 16)
    rng = np.random.default_rng(6)
    _warm(eng, rng, 7)
    acts = _plan_actions(eng, rng, H + K, n)
    live = eng.snapshot()
    la = eng.lookahead(acts[:H].contiguous(), leaf=True)
    leaf = EnvSnapshotCopy(la.leaf)
    # the clone: the roots stepped H + K steps in the live engine
    ref = []
    for t in range(H + K):
        eng.step(acts[t].contiguous())
        if t >= H:
            ref.append((eng.reward.clone(), eng.terminated.clone(), eng.obs().clone()))
    steps = la.steps.cpu().numpy()
    keep = torch.from_numpy(steps == H).to(eng.device)  # branches that ran the whole horizon: clones still live
    eng.restore(leaf.snap)
    for t in range(K):
        eng.step(acts[H + t].contiguous())
        r, te, o = ref[t]
        assert torch.equal(eng.reward[keep], r[keep]) and torch.equal(eng.terminated[keep], te[keep]), t
        assert torch.equal(eng.obs()[keep], o[keep]), t
    assert keep.any()
    eng.restore(live)
    eng.close()


class EnvSnapshotCopy:
    """A leaf snapshot detached from the Lookahead's storage (out= reuse would overwrite it)."""

    def __init__(self, snap):
        from carlabev_env_b200 import engine as E

        info = E.CbevSnapshotInfo()
        C.memmove(C.addressof(info), C.addressof(snap.info), C.sizeof(info))
        self.snap = E.EnvSnapshot(snap.data.clone(), info)


@pytest.mark.parametrize("R0", [0, 1])
def test_rows_taken_at_fewer_retreat_slots(R0):
    """Rows taken at R = 0 or 1 are roots after an append-only pool extension that raises R: the call from them equals
    restoring them and calling from the live envs."""
    import torch

    if R0 == 0:
        scenes = _scripted(12, kinds=[("lead_brake", 1 + i % 3) for i in range(12)])
    else:
        scenes = _scripted(12, kinds=[("jaywalk", 3)] * 12)
    n = 24
    eng = _engine(scenes, n, trajectory_steps=0)
    eng.reset(np.arange(n, dtype=np.int32) % len(scenes))
    rng = np.random.default_rng(9)
    _warm(eng, rng, 9)
    snap = eng.snapshot()
    assert snap.info.retreat_slots == R0
    walkers = _scripted(4, seed0=900, kinds=[("jaywalk", 3)] * 4)
    from carlabev_env_b200.pool import pack_pool

    eng.upload_pool(pack_pool(scenes + [_two_walkers(walkers[i], walkers[i + 1]) for i in range(0, 4, 2)]))
    assert eng.snapshot_row_bytes > snap.row_bytes
    roots = rng.integers(0, n, size=40)
    acts = _plan_actions(eng, rng, 20, 40)
    la = eng.lookahead(acts, source=snap, rows=roots, rewards=True, hero=True, obs=True, leaf=True)
    got, leaf = _results(la), la.leaf.data.clone()
    assert la.leaf.info.retreat_slots == 2 and la.leaf.row_bytes == eng.snapshot_row_bytes
    eng.restore(snap)
    ref = eng.lookahead(acts, env_ids=roots, rewards=True, hero=True, obs=True, leaf=True)
    _same_results(_results(ref), got, "grown pool")
    assert torch.equal(ref.leaf.data, leaf)
    eng.close()


def test_edge_roots():
    """Terminal roots (live and rows), out-of-range device roots and rows whose header scene lies outside the pool:
    steps = 0, the root's own row and window, or a zero window and an untouched (sentinel) leaf row."""
    import torch

    from carlabev_env_b200 import engine as E

    n = 16
    eng = _engine(_scripted(16), n, action_mode=E.ACTION_DISCRETE, discrete_table=TABLE,
                  reward_mode=E.REWARD_SHAPING, reward_params={"max_actions": 12})
    eng.reset(np.arange(n, dtype=np.int32))
    rng = np.random.default_rng(3)
    _warm(eng, rng, 5)
    bad = torch.tensor([-1, n, 0, 10 ** 6, 3, 7], dtype=torch.int32, device=eng.device)
    acts = _plan_actions(eng, rng, 6, 6)
    snap = eng.snapshot()
    la = eng.lookahead(acts, env_ids=bad, obs=True, leaf=True)
    la.leaf._buf.fill_(SENTINEL)
    la = eng.lookahead(acts, env_ids=bad, obs=True, leaf=True, out=la)
    steps = la.steps.cpu().numpy()
    ref = _leaf_reference(eng, snap, bad.cpu().numpy(), acts, steps, np.array([0, 0, 1, 0, 1, 1], dtype=bool))
    assert torch.equal(la.leaf.data, ref)
    assert steps[[0, 1, 3]].tolist() == [0, 0, 0] and not la.obs[[0, 1, 3]].any()
    assert (la.leaf.data[[0, 1, 3]] == SENTINEL).all()
    # rows as roots: out of range, and header scenes outside the pool
    rows = snap.data.clone()
    hdr = rows[:, :12].view(torch.int32)
    hdr[1, 0], hdr[2, 0] = -1, 10 ** 6
    forged = E.EnvSnapshot(rows, snap.info)
    roots = torch.tensor([0, 1, 2, -5, n, 4], dtype=torch.int32, device=eng.device)
    la = eng.lookahead(acts, source=forged, rows=roots, obs=True, leaf=True)
    la.leaf._buf.fill_(SENTINEL)
    la = eng.lookahead(acts, source=forged, rows=roots, obs=True, leaf=True, out=la)
    assert la.steps.cpu().tolist()[1:5] == [0, 0, 0, 0]
    assert not la.obs[1:5].any() and (la.leaf.data[1:5] == SENTINEL).all()
    live = eng.lookahead(acts[:, [0, 5]].contiguous(), env_ids=np.array([0, 4]), obs=True, leaf=True)
    assert torch.equal(la.obs[[0, 5]], live.obs) and torch.equal(la.leaf.data[[0, 5]], live.leaf.data)
    # every env truncated: terminal roots give steps = 0, their own window and exactly their own row
    _warm(eng, rng, 7)
    snap = eng.snapshot()
    assert snap.header()[:, 2].all()
    roots = rng.integers(0, n, size=24)
    acts = _plan_actions(eng, rng, 5, 24)
    for kw in (dict(env_ids=roots), dict(source=snap, rows=roots)):
        la = eng.lookahead(acts, obs=True, leaf=True, **kw)
        assert not la.steps.any()
        assert torch.equal(la.leaf.data, snap.data[torch.from_numpy(roots).to(eng.device)])
        assert torch.equal(la.obs, eng.obs()[torch.from_numpy(roots).to(eng.device)])
    eng.close()


def test_errors():
    import torch

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.pool import pack_pool

    n = 8
    scenes = _scripted(8)
    eng = _engine(scenes, n)
    other = _engine(scenes, n)
    for e in (eng, other):
        e.reset(np.arange(n, dtype=np.int32))
    acts = _plan_actions(eng, np.random.default_rng(0), 4, n)
    snap = eng.snapshot()
    with pytest.raises(ValueError, match="needs source="):
        eng.lookahead(acts, rows=np.arange(n))
    with pytest.raises(ValueError, match="exclusive"):
        eng.lookahead(acts, env_ids=np.arange(n), source=snap)
    with pytest.raises(ValueError, match=r"rows must lie in \[0, 8\)"):
        eng.lookahead(acts, source=snap, rows=np.arange(n) + 1)
    with pytest.raises(ValueError, match="another engine"):
        other.lookahead(acts, source=snap)
    # the C call: foreign rows are a state error, undersized or misaligned leaf buffers argument errors
    lib = eng.lib
    ret = torch.empty(n, dtype=torch.float64, device=eng.device)
    st = torch.empty(n, dtype=torch.int32, device=eng.device)
    o = E.CbevLookaheadOut(ret.data_ptr(), None, st.data_ptr(), None, None, None, None)
    buf = torch.empty(n * eng.snapshot_row_bytes + 64, dtype=torch.uint8, device=eng.device)
    info = E.CbevSnapshotInfo()

    def call(h, src, leaf_ptr, leaf_bytes):
        io = E.CbevLookaheadIo(C.pointer(src.info) if src else None, src._buf.data_ptr() if src else None, None,
                               None, 0, leaf_ptr, leaf_bytes, C.pointer(info))
        return lib.cbev_lookahead_ex(h.handle, C.byref(io), n, 4, acts.data_ptr(), 1.0, C.byref(o), h._stream())

    assert call(other, snap, None, 0) == 3
    assert call(eng, None, buf.data_ptr(), n * eng.snapshot_row_bytes - 1) == 1
    assert "leaf_rows holds" in lib.cbev_last_error().decode()
    assert call(eng, None, buf.data_ptr() + 8, buf.numel()) == 1
    assert "16-byte aligned" in lib.cbev_last_error().decode()
    assert call(eng, snap, buf.data_ptr(), buf.numel()) == 0
    torch.cuda.synchronize()
    # an ended pool epoch: before the next reset, and after it
    eng.invalidate()
    with pytest.raises(ValueError, match="epoch"):
        eng.lookahead(acts, source=snap)
    eng.upload_pool(pack_pool(scenes))
    eng.reset(np.arange(n, dtype=np.int32))
    with pytest.raises(ValueError, match="epoch"):
        eng.lookahead(acts, source=snap)
    assert call(eng, snap, None, 0) == 3
    eng.close()
    other.close()


def test_live_engine_is_untouched():
    """A call from rows with leaf rows leaves the live snapshot, ring, head and statistics byte-identical, and the
    engine then steps exactly as a twin that never planned."""
    from carlabev_env_b200 import engine as E

    n = 16
    engs = [_engine(_scripted(16), n, autoreset=E.AUTORESET_NEXT_STEP) for _ in range(2)]
    rngs = [np.random.default_rng(4), np.random.default_rng(4)]
    for e, r in zip(engs, rngs):
        e.reset(np.arange(n, dtype=np.int32))
        _warm(e, r, 9)
    eng, twin = engs
    snap = eng.snapshot()
    _warm(eng, rngs[0], 2)
    _warm(twin, rngs[1], 2)
    before = _live_state(eng)
    acts = _plan_actions(eng, np.random.default_rng(1), 16, 40)
    roots = np.random.default_rng(2).integers(0, n, size=40)
    la = eng.lookahead(acts, source=snap, rows=roots, rewards=True, hero=True, leaf=True)
    eng.lookahead(acts, source=la.leaf, leaf=True, obs=True)
    _same_state(before, _live_state(eng), "after the calls")
    _same_state(_live_state(twin), _live_state(eng), "against the twin", twin=True)
    for e, r in zip(engs, rngs):
        _warm(e, r, 3)
    _same_state(_live_state(twin), _live_state(eng), "twin, 3 steps later", twin=True)
    for e in engs:
        e.close()


def test_out_reuse_and_growth():
    import torch

    from carlabev_env_b200.pool import pack_pool

    scenes = _scripted(12, kinds=[("jaywalk", 3)] * 12)
    n = 16
    eng = _engine(scenes, n, trajectory_steps=0)
    eng.reset(np.arange(n, dtype=np.int32) % 12)
    rng = np.random.default_rng(12)
    _warm(eng, rng, 4)
    acts = _plan_actions(eng, rng, 6, n)
    la = eng.lookahead(acts, leaf=True)
    ptr, rb = la.leaf._buf.data_ptr(), la.leaf.row_bytes
    again = eng.lookahead(acts, leaf=True, out=la)
    assert again is la and la.leaf._buf.data_ptr() == ptr
    chained = eng.lookahead(acts, source=la.leaf, leaf=True, out=la)  # in place: roots and leaves share storage
    ref = eng.lookahead(acts, source=EnvSnapshotCopy(eng.lookahead(acts, leaf=True).leaf).snap, leaf=True)
    assert chained is la and torch.equal(la.leaf.data, ref.leaf.data)
    walkers = _scripted(2, seed0=900, kinds=[("jaywalk", 3)] * 2)
    eng.upload_pool(pack_pool(scenes + [_two_walkers(walkers[0], walkers[1])]))
    eng.lookahead(acts, leaf=True, out=la)  # R grew: new storage with the wider rows
    assert la.leaf.row_bytes > rb and la.leaf.row_bytes == eng.snapshot_row_bytes
    more = eng.lookahead(_plan_actions(eng, rng, 6, 3 * n), env_ids=rng.integers(0, n, 3 * n), leaf=True)
    assert more.leaf.n_rows == 3 * n  # the branch state grew with B
    eng.close()


@pytest.mark.parametrize("workload", ["c2", "c3"])
def test_scale(workload):
    """4096 branches on the c2 workload (lead_brake pool, continuous, float32 masks), every leaf row against stepping;
    8192 on a c3-style pool (25 live-stepped vehicles, discrete, uint8 masks), a seeded sample of 256."""
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
        eng = E.Engine(n, ring_slots=7, action_mode=E.ACTION_DISCRETE, discrete_table=TABLE[:5],
                       autoreset=E.AUTORESET_DISABLED, max_actors=25, trajectory_steps=0, seed=0, mask_dtype="uint8")
        eng.upload_map(load_town01_map(128))
        eng.upload_pool(pack_pool(scenes))
    eng.reset(np.arange(n, dtype=np.int32) % k)
    rng = np.random.default_rng(1)
    _warm(eng, rng, 10)
    if workload == "c2":
        _check_leaf(eng, rng, np.arange(n), 8)
    else:
        roots = np.arange(n)
        acts = _plan_actions(eng, rng, 8, n)
        snap = eng.snapshot()
        la = eng.lookahead(acts, env_ids=roots, leaf=True)
        sample = np.sort(np.random.default_rng(8).choice(n, size=256, replace=False))
        sel = torch.from_numpy(sample).cuda()
        steps = la.steps.cpu().numpy()[sample]
        ref = _leaf_reference(eng, snap, roots[sample], acts.index_select(1, sel).contiguous(), steps,
                              np.ones(256, dtype=bool))
        assert torch.equal(la.leaf.data.index_select(0, sel), ref)
        fr = eng.lookahead(acts, source=la.leaf, leaf=True)  # 8192 rows as roots
        assert fr.leaf.n_rows == n
    eng.close()

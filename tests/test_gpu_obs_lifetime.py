"""How long a returned observation stays valid, against a model of the ring's slot rule.

`RingModel` is the specification.  Every env has L ring slots; the window is slots head-F+1 .. head.  A step call moves
the head one slot on (from L-1 back to F-1) and writes each env's new frame at the head; an env reset in that call
(auto-reset under next_step or same_step) instead gets its reset frame in all F window slots.  A masked reset or a
restore writes the F window slots of its envs at the current head.  Every slot s written at or above the mirror
point M = L-F+1 is also written at s-M, so that the window is whole again after the wrap.

Two rules follow (`test_model_lifetime`): without resets a view stays intact for L-2F+1 further calls (the mirror
write of a head reaches the oldest slot of a window held from an earlier call after L-2F+2 calls), and any reset of env
e rewrites e's slots H-F+1 .. H at that call's head H, so every view of e that shares them changes.  Under same_step
that includes the window the previous call returned, for every env that ends.

The GPU tests hold the zero-copy view and a clone of every call's observation and check, at every later call, that
each view the model calls intact still equals its clone env by env, and that the bound is tight: some view differs
from its clone in the first call the model says it is overwritten.  At the make_env level the previous call's `obs`
(stacked or fused) and `final_obs` are checked after `step`, and INTEGRATION.md's same-step rollout loop is run."""
import numpy as np
import pytest

from test_gpu_same_step import _acts
from test_gpu_snapshot import _engine, _scripted


class RingModel:
    """Write versions of every (env, slot) of the ring: a view is intact while the versions of its slots are."""

    def __init__(self, F, L, n):
        self.F, self.L, self.n = F, L, n
        self.M = L - F + 1  # mirror point
        self.ver = np.zeros((n, L), dtype=np.int64)
        self.head = F - 1
        self.write(np.ones(n, bool), np.ones(n, bool))  # the first reset

    def _slots(self, reset):
        first = self.head - self.F + 1 if reset else self.head
        out = []
        for s in range(first, self.head + 1):
            out.append(s)
            if self.F > 1 and s >= self.M:
                out.append(s - self.M)
        return out

    def write(self, envs, reset):
        """A frame of each env in `envs` at the current head; `reset` [n] bool: a reset frame (all F window slots)."""
        for e in np.flatnonzero(envs):
            self.ver[e, self._slots(bool(reset[e]))] += 1

    def step(self, reset):
        """A step call: the head moves on, every env writes a frame, the envs of `reset` a reset frame."""
        self.head += 1
        if self.head >= self.L:
            self.head = self.F - 1
        self.write(np.ones(self.n, bool), reset)

    def window(self):
        """(head, versions [n, F]) of the current window."""
        return self.head, self.ver[:, self.head - self.F + 1: self.head + 1].copy()

    def intact(self, view):
        head, saved = view
        return (self.ver[:, head - self.F + 1: head + 1] == saved).all(axis=1)


def model_lifetime(F, L, calls=None):
    """The fewest further step calls (no resets) that any view stays intact for, over every head of 3 wraps."""
    m = RingModel(F, L, 1)
    held = [(0, m.window())]
    life = []
    for t in range(1, calls or 3 * L + 3):
        m.step(np.zeros(1, bool))
        keep = []
        for t0, v in held:
            if m.intact(v)[0]:
                keep.append((t0, v))
            else:
                life.append(t - t0 - 1)
        held = keep + [(t, m.window())]
    return min(life)


@pytest.mark.parametrize("F", [1, 2, 3, 4, 5])
def test_model_lifetime(F):
    """L - 2F + 1 further calls without resets; a reset rewrites the window slots of its envs at the call's head, among
    them F - 1 slots of the window the previous call returned."""
    for L in (2 * F - 1, 2 * F, 2 * F + 3, 64):
        assert model_lifetime(F, L) == L - 2 * F + 1, (F, L)
    # the lifetimes the docs state for the default ring (L >= 2F) and the minimum ring
    assert model_lifetime(4, 64) == 57 and model_lifetime(4, 8) == 1 and model_lifetime(4, 7) == 0
    assert model_lifetime(2, 3) == 0
    if F > 1:
        m = RingModel(F, 2 * F, 2)
        m.step(np.zeros(2, bool))
        prev = m.window()
        m.step(np.array([True, False]))  # env 0 is reset (same_step: in the call that ends its episode)
        assert m.intact(prev).tolist() == [False, True]


# ---- engine level --------------------------------------------------------------------------------------------------
FORMS = ("f32", "u8", "gray")
MODES = ("next_step", "same_step", "masked")


def _configs():
    out = []
    for F in (2, 4):
        for L in (2 * F - 1, 2 * F, 2 * F + 3, None):
            for mode in MODES:
                out.append((F, L, mode, FORMS[len(out) % 3], 16 + len(out) % 5))
    return out


CONFIGS = _configs()
DEFAULT_SLOTS = 20  # ring_budget_bytes of the default-ring configurations: the Engine's rule gives this many slots


def run_lifetime(F, L, mode, form, n, seed, max_calls=400):
    """Drive one engine until its ring wrapped 3 times and a reset landed in the mirror zone, checking every held view
    at every call.  Returns the counters."""
    from carlabev_env_b200 import engine as E

    scenes = _scripted(16)
    frame = {"f32": 6 * 96 * 96 * 4, "u8": 6 * 96 * 96, "gray": 96 * 96}[form]
    kw = dict(frame_stack=F, ring_slots=L, ring_budget_bytes=DEFAULT_SLOTS * n * frame,
              autoreset={"next_step": E.AUTORESET_NEXT_STEP, "same_step": E.AUTORESET_SAME_STEP,
                         "masked": E.AUTORESET_DISABLED}[mode])
    if form == "u8":
        kw["mask_dtype"] = "uint8"
    elif form == "gray":
        kw["obs_mode"] = E.OBS_GRAY
    eng = _engine(scenes, n, **kw)
    if L is None:
        assert eng.L == DEFAULT_SLOTS, eng.L
    L = eng.L
    eng.reset(np.arange(n, dtype=np.int32) % len(scenes))
    model = RingModel(F, L, n)
    c = dict(calls=0, wraps=0, resets=0, mirror_resets=0, checks=0, tight_ring=0, tight_reset=0, restores=0)
    held = []  # [call, model view, device view, clone, intact envs so far]
    rng = np.random.default_rng(seed)
    ep, k = np.zeros(n, np.int64), np.zeros(n, np.int64)
    pending = np.zeros(n, bool)  # next_step: ended in the last call, reset in the next

    def check(resetting):
        """Every held view the model calls intact equals its clone; count the views that differ in the first call
        the model calls them overwritten (by the head or mirror write, or by a reset of that env)."""
        keep = []
        for h in held:
            _, mv, view, clone, was = h
            now = model.intact(mv)
            diff = (view != clone).reshape(n, -1).any(1).cpu().numpy()
            bad = np.flatnonzero(now & diff)
            assert not len(bad), (F, L, mode, c["calls"], h[0], "a view the model calls intact changed", bad)
            first = was & ~now
            c["tight_ring"] += int((first & diff & ~resetting).sum())
            c["tight_reset"] += int((first & diff & resetting).sum())
            c["checks"] += 1
            h[4] = now
            if now.any():
                keep.append(h)
        held[:] = keep

    def hold():
        view = eng.obs()
        held.append([c["calls"], model.window(), view, view.clone(), np.ones(n, bool)])
        assert eng.head == model.head, (eng.head, model.head)

    hold()
    while c["calls"] < max_calls and not (c["wraps"] >= 3 and c["mirror_resets"] >= 1 and c["restores"] >= 1):
        c["calls"] += 1
        h0 = eng.head
        eng.step(_acts(False, 0, ep, k, seed))
        ended = (eng.terminated | eng.truncated).cpu().numpy().astype(bool)
        resetting = pending.copy() if mode == "next_step" else ended if mode == "same_step" else np.zeros(n, bool)
        model.step(resetting)
        c["wraps"] += int(eng.head < h0)
        c["resets"] += int(resetting.sum())
        c["mirror_resets"] += int(resetting.sum()) * int(model.head >= model.M)
        check(resetting)
        hold()
        k += 1
        ep[ended] += 1
        k[ended] = 0
        if mode == "next_step":
            pending = ended
        if mode == "masked":  # every env that ended, and every fifth call a few more
            mask = ended | ((rng.random(n) < 0.2) if c["calls"] % 5 == 0 else False)
            if mask.any():
                c["calls"] += 1
                eng.reset(np.arange(n, dtype=np.int32) % len(scenes), mask)
                model.write(mask, mask)
                c["resets"] += int(mask.sum())
                c["mirror_resets"] += int(mask.sum()) * int(model.head >= model.M)
                check(mask)
                hold()
        if c["calls"] >= L and c["restores"] == 0:  # clone envs 2 and 3 into envs 0 and 1
            c["calls"] += 1
            snap = eng.snapshot([2, 3])
            eng.restore(snap, env_ids=[0, 1])
            done = snap.header()[:, 2].cpu().numpy() != 0
            mask = np.zeros(n, bool)
            mask[:2] = True
            model.write(mask, mask)
            if mode == "next_step":
                pending[:2] = done
            c["restores"] += 1
            check(mask)
            hold()
    eng.close()
    return c


@pytest.mark.gpu
@pytest.mark.timeout(600)
@pytest.mark.parametrize("F,L,mode,form,n", CONFIGS,
                         ids=[f"F{F}-L{L or 'default'}-{m}-{fo}" for F, L, m, fo, _ in CONFIGS])
def test_views_last_as_the_model_says(F, L, mode, form, n):
    c = run_lifetime(F, L, mode, form, n, seed=CONFIGS.index((F, L, mode, form, n)))
    print(F, L, mode, form, n, c)
    assert c["wraps"] >= 3 and c["mirror_resets"] >= 1 and c["restores"] == 1, c
    assert c["tight_ring"] >= 1, ("no view changed in the first call the head or mirror write reached it", c)
    assert c["tight_reset"] >= 1, ("no view changed in the first call a reset reached it", c)


# ---- make_env level ------------------------------------------------------------------------------------------------
VEC = [(fusion, mode) for fusion in ("stack", "vehicle_temporal", "vehicle_weighted")
       for mode in ("next_step", "same_step")]


@pytest.mark.gpu
@pytest.mark.timeout(600)
@pytest.mark.parametrize("fusion,mode", VEC, ids=[f"{f}-{m}" for f, m in VEC])
def test_make_env_previous_obs_and_rollout_loop(fusion, mode):
    """After `step`, the previous call's `obs` is intact for every env that `step` did not reset (stacked) or for
    every env (fused: two buffers in turn), and the previous call's `final_obs` rows stay intact for the envs that do
    not end again.  INTEGRATION.md's rollout loop (obs copied into the buffer before `step`) stores exactly what a
    loop that clones every returned observation stores; storing the previous `obs` after `step` instead gives the same
    for fused observations and differs for stacked ones only in envs that `step` reset."""
    import torch

    from carlabev_env_b200.config import EnvConfig, RunConfig
    from carlabev_env_b200.vector_env import make_env

    cfg = RunConfig(env=EnvConfig(action_mode="continuous", temporal_fusion_mode=fusion), num_envs=24)
    envs = make_env(cfg, scenes=_scripted(16), autoreset=mode, ring_budget_bytes=32 << 20)
    N, T = envs.num_envs, 48
    F, L = envs.engine.F, envs.engine.L
    assert L == 2 * F  # the default rule's floor at this budget: the previous window outlives one call exactly
    obs, _ = envs.reset(options={"scene": "pool"})
    obs_buf = torch.empty((T, *obs.shape), dtype=obs.dtype, device=obs.device)
    cloned, after = [], []  # what a cloning loop stores; the previous obs stored after the step
    ep, k = np.zeros(N, np.int64), np.zeros(N, np.int64)
    pending = np.zeros(N, bool)
    prev_final = None
    c = dict(reset_envs=0, reset_changed=0, final_kept=0)
    for t in range(T):
        obs_buf[t] = obs  # INTEGRATION.md: before the step
        cloned.append(obs.clone())
        prev = obs
        obs, rew, term, trunc, infos = envs.step(_acts(False, 0, ep, k, VEC.index((fusion, mode)), host=True))
        ended = (term | trunc).cpu().numpy()
        reset = ended if mode == "same_step" else pending
        after.append(prev.clone())
        same = (prev == cloned[t]).reshape(N, -1).all(1).cpu().numpy()
        c["reset_envs"] += int(reset.sum())
        if fusion == "stack":
            assert same[~reset].all(), (t, "previous obs changed in envs step did not reset", np.flatnonzero(~same))
            c["reset_changed"] += int((~same[reset]).sum())
        else:
            assert same.all(), (t, "previous fused obs changed", np.flatnonzero(~same))
        if prev_final is not None:
            fin, fin_clone, fin_ended = prev_final
            keep = fin_ended & ~ended
            assert torch.equal(fin[torch.from_numpy(keep).cuda()], fin_clone[torch.from_numpy(keep).cuda()]), t
            c["final_kept"] += int(keep.sum())
        if mode == "same_step" and ended.any():
            prev_final = (infos["final_obs"], infos["final_obs"].clone(), ended)
        k += 1
        ep[ended] += 1
        k[ended] = 0
        pending = ended
    envs.close()
    for t in range(T):
        assert torch.equal(obs_buf[t], cloned[t]), (t, "the INTEGRATION loop stored another observation")
    assert c["reset_envs"] >= 4, c
    if fusion == "stack":  # the reset frames rewrite F - 1 slots of the window the previous call returned
        assert c["reset_changed"] >= 1, c
    else:
        assert all(torch.equal(a, b) for a, b in zip(after, cloned)), "fused obs stored after the step changed"
    if mode == "same_step":
        assert c["final_kept"] >= 1, c

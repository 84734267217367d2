"""Every pair of configuration settings against the oracle, with the full step outputs and action repeat.

`ROWS` is a pairwise covering array over the axes of `AXES`: for any two axes, every pair of values that some valid
configuration can hold together appears in at least one row.  It is the checked-in output of `generate()`, a greedy
covering-array generator (below), so the rows are fixed and a change to the axes or rules shows up as a diff of the
table; `test_rows_are_the_generator_output` keeps the two in step.

Each row runs `run_row` on the GPU: a small batch (12-24 envs, some not a multiple of 16) driven for 80-120 agent
steps, every env compared with `OracleEnv` on every step -- the observation in the row's form (stacked, fused, uint8,
gray or the raw frame), reward, flags, cause, the whole hero block, actor poses, the episode row of every terminal
step, the scene of every device auto-reset or the observation of every masked reset, and at the end the statistics
vector.  Rows at action repeat K > 1 step the oracle with `oracle_pool`'s ("repeat", (action, K)) command.  In the
same_step rows a call that ends an env is checked against the oracle's terminal sub-step (the terminal window through
`final_obs`, fused in the fusion rows) and, in that same call, against the oracle reset on the scene the device drew:
observation, actor poses and the snapshot header's scene; the `final_obs` rows of the envs that did not end must keep
their contents.  The `ring_slots` column alternates the Engine's default ring and the smallest one, 2F - 1 slots,
whose rows must put a reset frame in the mirror zone.

Axes and the values that are not obvious from their names:
  resize   which resize branch of the raster kernels the observation takes (`OBS_SIZE`): `fast96` is k_render's
           128 -> 96 x 96; `area` an INTER_AREA table; `half` the 2x integer path; `copy` obs = fov; `enlarge`
           OpenCV's bilinear branch; `block83` k_render_any's 8:3 block shortcut (taken only with the FOV mask off);
           `nonsquare` a table with different factors per axis; `raw` the (size, size, 3) frame.
  anchor   the centre, (0.5, 0.75), the corner (0, 1) (ego square on the frame's edge) and (0.95, 0.3), whose crop
           sides are odd at every scale (149 / 301 / 603; the centre's are odd at 64 and 256: 91 / 363).
  actors   trajectory tables (1024 steps), a table -> live hand-over at step 40, or live stepping with more than 8
           actor slots (the 32-lane groups of the sim kernels).
  repeat   1 or K > 1: 3, except every fourth repeat row, at 4 or 8 in turn.
  path     `Engine.step` with device actions, or `cbev_step_host_ex` with pinned host actions and the host mirrors of
           reward, flags and episode rows, as `vector_env.py` drives it.
A setting that a configuration does not have is None: no mask mode for gray and RGB, no fusion outside the semantic
masks, no frame stack for the raw frame.

The scene pools mix rdm scenes with up to 15 vehicles (so the live rows take the 32-lane path) and, at scale 128 only
(quirk C-11), lead_brake, jaywalk and red_light_runner scenes.  Envs drive by index (`test_gpu_reward_params.drive`):
route pursuit, full throttle, a lateral bias onto the sidewalk and braking into reverse, so that episodes end by
success, collision, off-road and, in the shaping rows with a short `max_actions`, truncation.  No row passes without
compared terminal episodes, an auto-reset in the next_step rows, MIN_EPISODES same-step resets in the same_step rows
and an episode that ends inside a repeat in the repeat rows (reset in that call in the same_step ones)."""
import itertools

import numpy as np
import pytest

from golden_util import load_map

AXES = {
    "size": (64, 128, 256),
    "resize": ("fast96", "area", "half", "copy", "enlarge", "block83", "nonsquare", "raw"),
    "obs": ("f32", "u8", "gray", "rgb"),
    "mask": ("binary", "2-class", "4-class", "5-class", "6-class", "7-class"),
    "anchor": ((0.5, 0.5), (0.5, 0.75), (0.0, 1.0), (0.95, 0.3)),
    "fov": (False, True),
    "fusion": ("stack", "vehicle_temporal", "vehicle_weighted"),
    "frame_stack": (3, 4, 5),
    "actions": ("continuous", "discrete9", "discrete13"),
    "reward": ("carl", "shaping"),
    "actors": ("tables", "handover", "live"),
    "autoreset": ("next_step", "same_step", "disabled"),
    "repeat": (1, 3),
    "path": ("device", "host"),
}
# observation (h, w) of each resize branch per map scale; `fast96` exists at 128 only, `enlarge` not at 256 (the
# engine takes at most 256 per side)
OBS_SIZE = {
    "fast96": {128: (96, 96)},
    "area": {64: (48, 48), 128: (84, 84), 256: (84, 84)},
    "half": {64: (32, 32), 128: (64, 64), 256: (128, 128)},
    "copy": {64: (64, 64), 128: (128, 128), 256: (256, 256)},
    "enlarge": {64: (96, 96), 128: (160, 160)},
    "block83": {64: (24, 24), 128: (48, 48), 256: (96, 96)},
    "nonsquare": {64: (48, 40), 128: (112, 100), 256: (100, 60)},
}
OPTIONAL = ("mask", "fusion", "frame_stack")  # the axes that some configurations do not have (None)
VEHICLE_MASKS = ("4-class", "5-class", "6-class", "7-class")  # the mask modes with a vehicle channel (fusion)
ACTION_PROFILE = {"continuous": "continuous_gsb_v1", "discrete9": "discrete9_v1", "discrete13": "discrete13_v1"}
TRAJECTORY_STEPS = {"tables": 1024, "handover": 40, "live": 0}
N_ENVS = (12, 16, 19, 24, 13, 20)  # by row index: some batches are not a multiple of the 16 envs of a CTA
SHORT_MAX_ACTIONS = 45  # every other shaping row: truncations


def _conflict(r):
    """Whether the partial row `r` (axis -> value) breaks a rule; rules whose axes are not all set are skipped."""
    def has(*keys):
        return all(k in r for k in keys)

    if any(v is None for k, v in r.items() if k not in OPTIONAL):
        return True
    if has("size", "resize") and r["resize"] != "raw" and r["size"] not in OBS_SIZE[r["resize"]]:
        return True
    if has("obs", "resize") and (r["obs"] == "rgb") != (r["resize"] == "raw"):  # the raw frame is not resized
        return True
    masks = r.get("obs") in ("f32", "u8")
    if has("obs", "mask") and (r["mask"] is not None) != masks:
        return True
    if has("obs", "fusion") and (r["fusion"] is not None) != masks:
        return True
    if has("obs", "frame_stack") and (r["frame_stack"] is None) != (r["obs"] == "rgb"):  # raw frames: F = 1
        return True
    if has("fusion", "mask") and r["fusion"] not in (None, "stack") and r["mask"] not in VEHICLE_MASKS:
        return True
    if has("fusion", "frame_stack") and r["fusion"] not in (None, "stack") and r["frame_stack"] < 3:
        return True
    if has("obs", "size", "resize") and r["resize"] in OBS_SIZE and r["size"] in OBS_SIZE[r["resize"]]:
        h, w = OBS_SIZE[r["resize"]][r["size"]]
        if h * w % (4 if r["obs"] == "f32" else 16):  # 16-byte stores of the planes
            return True
    return False


def _completable(r):
    """Whether the partial row `r` has a completion that breaks no rule (depth-first over the unset axes)."""
    if _conflict(r):
        return False
    for ax, dom in AXES.items():
        if ax not in r:
            return any(_completable({**r, ax: v}) for v in dom + (None,))
    return True


def _pairs(row):
    """The (axis, value, axis, value) pairs of a row, None values left out."""
    items = [(a, row[a]) for a in AXES if row.get(a) is not None]
    return {(a, v, b, w) for (a, v), (b, w) in itertools.combinations(items, 2)}


def allowed_pairs():
    out = set()
    for a, b in itertools.combinations(AXES, 2):
        out |= {(a, v, b, w) for v in AXES[a] for w in AXES[b] if _completable({a: v, b: w})}
    return out


def _key(pair):
    a, v, b, w = pair
    return list(AXES).index(a), AXES[a].index(v), list(AXES).index(b), AXES[b].index(w)


def generate():
    """Greedy pairwise covering array (AETG-style, deterministic).  Rows start from three seeds -- the 8:3 shortcut
    with the FOV mask off at every scale, the only configuration that takes it -- and then from the first uncovered
    pair in axis / value order.  Every other axis takes, in axis order, the value that completes to a valid row and
    covers the most uncovered pairs with the values already set (ties: the value earlier rows used least, then the
    first in `AXES` order, None last), so the rows that only fill the last pairs still spread over every value.  A row
    then takes its N, its agent steps and, in the shaping rows, every other one a short `max_actions`; every fourth row
    at repeat 3 is moved to 4 or 8 in turn; the rows with a frame stack alternate between the Engine's default ring
    (None) and the smallest ring the ABI takes, 2F - 1 slots."""
    uncovered = allowed_pairs()
    seeds = [dict(size=s, resize="block83", fov=False) for s in AXES["size"]]
    rows = []
    used = {}  # (axis, value) -> rows so far
    while uncovered or seeds:
        if seeds:
            row = seeds.pop(0)
        else:
            a, v, b, w = min(uncovered, key=_key)
            row = {a: v, b: w}
        for ax, dom in AXES.items():
            if ax in row:
                continue
            best = None
            for v in dom + (None,):
                cand = {**row, ax: v}
                if not _completable(cand):
                    continue
                score = (len(_pairs(cand) & uncovered), -used.get((ax, v), 0))
                if best is None or score > best[0]:
                    best = (score, v)
            row[ax] = best[1]
        uncovered -= _pairs(row)
        for ax, v in row.items():
            used[ax, v] = used.get((ax, v), 0) + 1
        rows.append({ax: row[ax] for ax in AXES})
    shaping = repeats = stacked = 0
    for i, row in enumerate(rows):
        row["n_envs"] = N_ENVS[i % len(N_ENVS)]
        row["steps"] = 80 + (7 * i) % 41
        row["max_actions"] = None
        if row["reward"] == "shaping":
            row["max_actions"] = SHORT_MAX_ACTIONS if shaping % 2 == 0 else None
            shaping += 1
        if row["repeat"] > 1:
            if repeats % 4 == 3:
                row["repeat"] = (4, 8)[(repeats // 4) % 2]
            repeats += 1
        row["ring_slots"] = None
        if row["frame_stack"] is not None:
            row["ring_slots"] = 2 * row["frame_stack"] - 1 if stacked % 2 else None
            stacked += 1
    return rows


# ring_slots: None is the Engine's rule at `run_row`'s 64 MB budget (2F..64 slots); 2F - 1 puts the head in the mirror
# zone (slots >= L - F + 1) F - 1 calls out of F, so that resets land there often
COLUMNS = tuple(AXES) + ("n_envs", "steps", "max_actions", "ring_slots")
ROWS = [  # generate(), one tuple per row in COLUMNS order
    (64, 'block83', 'f32', 'binary', (0.5, 0.5), False, 'stack', 3, 'continuous', 'carl', 'tables', 'next_step', 1, 'device', 12, 80, None, None),
    (128, 'block83', 'u8', '2-class', (0.5, 0.75), False, 'stack', 4, 'discrete9', 'shaping', 'handover', 'same_step', 3, 'host', 16, 87, 45, 7),
    (256, 'block83', 'gray', None, (0.0, 1.0), False, None, 5, 'discrete13', 'carl', 'live', 'disabled', 3, 'device', 19, 94, None, None),
    (64, 'area', 'u8', '4-class', (0.95, 0.3), True, 'vehicle_temporal', 5, 'continuous', 'shaping', 'live', 'next_step', 1, 'host', 24, 101, None, 9),
    (64, 'half', 'gray', None, (0.5, 0.75), True, None, 3, 'discrete9', 'carl', 'handover', 'disabled', 1, 'device', 13, 108, None, None),
    (64, 'copy', 'f32', '5-class', (0.0, 1.0), True, 'vehicle_weighted', 4, 'discrete13', 'shaping', 'tables', 'same_step', 3, 'host', 20, 115, 45, 7),
    (64, 'enlarge', 'f32', '6-class', (0.95, 0.3), False, 'vehicle_temporal', 3, 'discrete9', 'carl', 'tables', 'same_step', 4, 'device', 12, 81, None, None),
    (64, 'nonsquare', 'u8', '7-class', (0.5, 0.5), True, 'vehicle_weighted', 5, 'discrete9', 'carl', 'handover', 'next_step', 3, 'host', 16, 88, None, 9),
    (64, 'raw', 'rgb', None, (0.5, 0.5), False, None, None, 'discrete13', 'shaping', 'live', 'disabled', 1, 'device', 19, 95, None, None),
    (64, 'area', 'f32', '2-class', (0.5, 0.75), True, 'stack', 5, 'discrete13', 'carl', 'tables', 'disabled', 1, 'device', 24, 102, None, None),
    (128, 'fast96', 'gray', None, (0.95, 0.3), True, None, 4, 'continuous', 'carl', 'handover', 'disabled', 1, 'host', 13, 109, None, 7),
    (128, 'area', 'gray', None, (0.5, 0.5), False, None, 3, 'discrete13', 'shaping', 'live', 'same_step', 3, 'host', 20, 116, 45, None),
    (128, 'half', 'f32', '4-class', (0.0, 1.0), False, 'vehicle_weighted', 3, 'continuous', 'shaping', 'tables', 'next_step', 3, 'device', 12, 82, None, 5),
    (128, 'copy', 'u8', 'binary', (0.5, 0.75), True, 'stack', 5, 'continuous', 'shaping', 'live', 'same_step', 1, 'device', 16, 89, 45, None),
    (128, 'enlarge', 'u8', '5-class', (0.0, 1.0), False, 'vehicle_temporal', 4, 'discrete13', 'carl', 'handover', 'next_step', 1, 'device', 19, 96, None, 7),
    (128, 'nonsquare', 'gray', None, (0.95, 0.3), False, None, 4, 'discrete13', 'shaping', 'tables', 'next_step', 1, 'device', 24, 103, None, None),
    (128, 'raw', 'rgb', None, (0.5, 0.75), True, None, None, 'discrete9', 'carl', 'handover', 'next_step', 8, 'host', 13, 110, None, None),
    (128, 'fast96', 'u8', '6-class', (0.5, 0.5), True, 'vehicle_temporal', 3, 'discrete13', 'shaping', 'live', 'disabled', 3, 'host', 20, 117, 45, 5),
    (128, 'fast96', 'f32', '7-class', (0.0, 1.0), False, 'stack', 4, 'discrete9', 'shaping', 'live', 'same_step', 1, 'device', 12, 83, None, None),
    (256, 'area', 'f32', 'binary', (0.95, 0.3), True, 'stack', 4, 'discrete9', 'shaping', 'handover', 'same_step', 3, 'host', 16, 90, 45, 7),
    (256, 'half', 'u8', '2-class', (0.5, 0.5), False, 'stack', 3, 'continuous', 'carl', 'tables', 'next_step', 1, 'host', 19, 97, None, None),
    (256, 'copy', 'gray', None, (0.5, 0.75), False, None, 3, 'discrete9', 'carl', 'handover', 'disabled', 3, 'host', 24, 104, None, 5),
    (256, 'nonsquare', 'f32', '4-class', (0.5, 0.75), True, 'vehicle_temporal', 4, 'continuous', 'carl', 'live', 'same_step', 1, 'device', 13, 111, None, None),
    (256, 'raw', 'rgb', None, (0.0, 1.0), True, None, None, 'continuous', 'shaping', 'tables', 'same_step', 4, 'host', 20, 118, None, None),
    (256, 'half', 'u8', '5-class', (0.95, 0.3), False, 'vehicle_weighted', 5, 'continuous', 'carl', 'live', 'disabled', 1, 'device', 12, 84, None, 9),
    (256, 'copy', 'f32', '6-class', (0.5, 0.5), True, 'vehicle_weighted', 4, 'continuous', 'shaping', 'handover', 'next_step', 1, 'host', 16, 91, 45, None),
    (256, 'block83', 'u8', '7-class', (0.95, 0.3), True, 'vehicle_temporal', 3, 'discrete13', 'carl', 'tables', 'disabled', 3, 'device', 19, 98, None, 5),
    (128, 'fast96', 'f32', 'binary', (0.0, 1.0), False, 'stack', 5, 'discrete13', 'shaping', 'tables', 'next_step', 3, 'host', 24, 105, None, None),
    (128, 'fast96', 'u8', '2-class', (0.5, 0.75), False, 'stack', 5, 'discrete9', 'carl', 'live', 'same_step', 1, 'device', 13, 112, None, 9),
    (128, 'fast96', 'f32', '4-class', (0.5, 0.5), True, 'vehicle_weighted', 5, 'discrete9', 'shaping', 'handover', 'disabled', 3, 'host', 20, 119, 45, None),
    (128, 'fast96', 'u8', '5-class', (0.5, 0.5), False, 'stack', 3, 'discrete9', 'carl', 'tables', 'next_step', 1, 'device', 12, 85, None, 5),
    (64, 'area', 'f32', '5-class', (0.0, 1.0), True, 'vehicle_weighted', 4, 'continuous', 'shaping', 'handover', 'same_step', 8, 'host', 16, 92, None, None),
    (64, 'area', 'u8', '6-class', (0.5, 0.75), False, 'vehicle_weighted', 5, 'discrete13', 'carl', 'live', 'disabled', 1, 'device', 19, 99, None, 9),
    (256, 'area', 'f32', '7-class', (0.5, 0.75), True, 'vehicle_temporal', 3, 'continuous', 'shaping', 'tables', 'next_step', 3, 'host', 24, 106, 45, None),
    (64, 'half', 'u8', 'binary', (0.95, 0.3), False, 'stack', 4, 'discrete13', 'carl', 'handover', 'same_step', 1, 'device', 13, 113, None, 7),
    (256, 'half', 'f32', '6-class', (0.0, 1.0), True, 'vehicle_temporal', 5, 'discrete9', 'shaping', 'live', 'disabled', 3, 'host', 20, 120, None, None),
    (64, 'half', 'u8', '7-class', (0.95, 0.3), False, 'vehicle_temporal', 3, 'continuous', 'carl', 'tables', 'next_step', 1, 'device', 12, 86, None, 5),
    (256, 'copy', 'f32', '2-class', (0.95, 0.3), True, 'stack', 4, 'discrete9', 'shaping', 'handover', 'same_step', 3, 'host', 16, 93, 45, None),
    (64, 'copy', 'u8', '4-class', (0.5, 0.5), False, 'vehicle_temporal', 5, 'discrete13', 'carl', 'live', 'disabled', 1, 'device', 19, 100, None, 9),
    (256, 'copy', 'f32', '7-class', (0.0, 1.0), True, 'vehicle_weighted', 3, 'continuous', 'shaping', 'tables', 'next_step', 4, 'host', 24, 107, None, None),
    (64, 'enlarge', 'gray', None, (0.5, 0.5), True, None, 5, 'continuous', 'shaping', 'live', 'disabled', 1, 'host', 13, 114, 45, 9),
    (64, 'enlarge', 'u8', 'binary', (0.5, 0.75), False, 'stack', 4, 'discrete9', 'carl', 'handover', 'disabled', 3, 'device', 20, 80, None, None),
    (128, 'enlarge', 'f32', '2-class', (0.0, 1.0), False, 'stack', 3, 'discrete13', 'carl', 'tables', 'same_step', 1, 'device', 12, 87, None, 5),
    (64, 'enlarge', 'u8', '4-class', (0.95, 0.3), True, 'vehicle_weighted', 4, 'discrete9', 'shaping', 'handover', 'next_step', 3, 'host', 16, 94, None, None),
    (128, 'enlarge', 'f32', '7-class', (0.5, 0.5), False, 'vehicle_temporal', 5, 'discrete13', 'carl', 'live', 'same_step', 1, 'device', 19, 101, None, 9),
    (256, 'block83', 'u8', '4-class', (0.5, 0.75), True, 'vehicle_weighted', 3, 'continuous', 'shaping', 'tables', 'next_step', 3, 'host', 24, 108, 45, None),
    (256, 'block83', 'f32', '5-class', (0.5, 0.75), False, 'vehicle_temporal', 4, 'discrete9', 'carl', 'handover', 'same_step', 1, 'device', 13, 115, None, 7),
    (256, 'block83', 'u8', '6-class', (0.0, 1.0), True, 'stack', 5, 'discrete13', 'shaping', 'live', 'disabled', 8, 'host', 20, 81, None, None),
    (64, 'nonsquare', 'f32', 'binary', (0.0, 1.0), False, 'stack', 3, 'continuous', 'carl', 'tables', 'disabled', 1, 'device', 12, 88, None, 5),
    (128, 'nonsquare', 'u8', '2-class', (0.95, 0.3), True, 'stack', 4, 'discrete9', 'shaping', 'handover', 'next_step', 3, 'host', 16, 95, 45, None),
    (256, 'nonsquare', 'f32', '5-class', (0.5, 0.5), False, 'vehicle_weighted', 5, 'discrete13', 'carl', 'live', 'same_step', 1, 'device', 19, 102, None, 9),
    (64, 'nonsquare', 'u8', '6-class', (0.95, 0.3), True, 'vehicle_temporal', 3, 'continuous', 'shaping', 'tables', 'next_step', 3, 'host', 24, 109, None, None),
    (128, 'raw', 'rgb', None, (0.95, 0.3), False, None, None, 'discrete9', 'carl', 'handover', 'same_step', 1, 'device', 13, 116, None, None),
    (256, 'area', 'f32', '4-class', (0.5, 0.5), True, 'stack', 4, 'discrete13', 'shaping', 'live', 'disabled', 3, 'host', 20, 82, 45, 7),
]


def _row(i):
    return dict(zip(COLUMNS, ROWS[i]))


def _scene_pool(size, anchor):
    """rdm scenes with 0-15 vehicles (at least one with more than 8 actors: the live rows take the 32-lane groups);
    at scale 128 also lead_brake, jaywalk and red_light_runner (the scripted kinds exist there only, quirk C-11).
    Scenes are built with the crop of `anchor` as the map padding, as the env builds them."""
    from carlabev_env_b200 import scenes as S
    from oracle import raster

    key = (size, anchor)
    if key in _POOLS:
        return _POOLS[key]
    cls = load_map(size)
    pad = raster.FovGeometry(size, *anchor).pad
    base = 1000 * size + 100 * AXES["anchor"].index(anchor)
    veh = (14, 3, 9, 0, 15, 6, 11, 2, 12, 5, 15, 8)
    reqs = [dict(scene="rdm", num_vehicles=v, route_dist_range=[30, 90], scene_seed=base + i) for i, v in enumerate(veh)]
    if size == 128:
        reqs = reqs[:8]
        reqs += [dict(scene="lead_brake", level=1 + i, scene_seed=base + 20 + i) for i in range(2)]
        reqs += [dict(scene="jaywalk", level=2 + i, scene_seed=base + 30 + i) for i in range(2)]
        reqs += [dict(scene="red_light_runner", scene_seed=base + 40 + i) for i in range(2)]
        scenes = [S.build_scene(r, cls_map=cls, pad=pad) for r in reqs]
    else:
        scenes = [sc for sc in S.build_pool(reqs, pad=pad, size=size, skip_invalid=True, workers=1) if sc is not None]
    assert len(scenes) >= 4 and max(len(sc["act_kind"]) for sc in scenes) > 8, (key, len(scenes))
    _POOLS[key] = scenes
    return scenes


_POOLS = {}


def engine_args(row):
    """Engine keyword arguments of a row (without the pool-dependent max_actors)."""
    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.config import ACTION_PROFILES

    obs = row["obs"]
    table = ACTION_PROFILES[ACTION_PROFILE[row["actions"]]].get("discrete_actions")
    return dict(obs_mode={"f32": E.OBS_SEMANTIC, "u8": E.OBS_SEMANTIC, "gray": E.OBS_GRAY, "rgb": E.OBS_RGB}[obs],
                mask_dtype="uint8" if obs == "u8" else "float32", mask_mode=row["mask"] or "6-class",
                frame_stack=row["frame_stack"] or 1, size=row["size"],
                obs_size=OBS_SIZE[row["resize"]][row["size"]] if obs != "rgb" else (96, 96), anchor=row["anchor"],
                action_mode=E.ACTION_CONTINUOUS if table is None else E.ACTION_DISCRETE, discrete_table=table,
                reward_mode=E.REWARD_SHAPING if row["reward"] == "shaping" else E.REWARD_CARL,
                reward_params={"max_actions": row["max_actions"]} if row["max_actions"] else None,
                autoreset={"next_step": E.AUTORESET_NEXT_STEP, "same_step": E.AUTORESET_SAME_STEP,
                           "disabled": E.AUTORESET_DISABLED}[row["autoreset"]],
                trajectory_steps=TRAJECTORY_STEPS[row["actors"]], ring_slots=row.get("ring_slots"))


def oracle_args(row):
    """OracleEnv keyword arguments of a row (without the map scale, which OraclePool takes)."""
    profile = ACTION_PROFILE[row["actions"]]
    return dict(obs_mode={"f32": "bev_semantic", "u8": "bev_semantic", "gray": "bev_gray", "rgb": "bev_raw"}[row["obs"]],
                semantic_mask_ch=row["mask"] or "6-class", frame_stack=row["frame_stack"] or 1,
                obs_size=OBS_SIZE[row["resize"]][row["size"]] if row["obs"] != "rgb" else (96, 96),
                action_mode="continuous" if row["actions"] == "continuous" else "discrete", action_profile=profile,
                reward_mode=row["reward"], reward_params={"max_actions": row["max_actions"]} if row["max_actions"] else None,
                anchor=row["anchor"], fov_masked=row["fov"], temporal_fusion_mode=row["fusion"] or "stack")


def run_row(row, seed=23):
    """Engine vs oracle on every env of the row's batch, every agent step (see the module doc).  Returns the counters."""
    import torch

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.config import ACTION_PROFILES
    from carlabev_env_b200.fovmask import corner_mask
    from carlabev_env_b200.pool import pack_pool
    from oracle_pool import OraclePool
    from test_gpu_action_repeat import _stats_from_rows
    from test_gpu_reward_params import drive
    from test_gpu_scale import POSE_TOL, _check_episode, _check_hero, autoreset_scene

    size, n, K, steps = row["size"], row["n_envs"], row["repeat"], row["steps"]
    scenes = _scene_pool(size, row["anchor"])
    S = len(scenes)
    amax = max(len(sc["act_kind"]) for sc in scenes)
    kw = engine_args(row)
    traj = kw["trajectory_steps"]
    eng = E.Engine(n, max_actors=amax, seed=seed, ring_budget_bytes=64 << 20, **kw)
    eng.upload_map(load_map(size))
    eng.upload_pool(pack_pool(scenes))
    if row["fov"]:
        eng.upload_fov_mask(corner_mask(size, 0.5))
    if K > 1:
        eng.set_action_repeat(K)
    eng.reset(torch.arange(n, dtype=torch.int32) % S)
    fuse = row["fusion"] if row["fusion"] not in (None, "stack") else None
    next_step = row["autoreset"] == "next_step"
    same_step = row["autoreset"] == "same_step"
    host = row["path"] == "host"
    F = eng.F
    mirror = eng.L - F + 1 if F > 1 else eng.L + 1  # heads from here on also write slot head - mirror
    table = ACTION_PROFILES[ACTION_PROFILE[row["actions"]]].get("discrete_actions")
    table = None if table is None else np.asarray(table, dtype=np.float32)
    u8 = row["obs"] == "u8"

    def observe():
        return (eng.fuse(fuse) if fuse else eng.obs()).cpu().numpy()

    def same_obs(got, ref):
        ref = ref[0] if row["obs"] == "rgb" else ref  # the raw frame has no frame stack
        if u8 and fuse != "vehicle_weighted":  # 0 / 1 bytes against the oracle's 0.0 / 1.0 floats
            assert np.isin(ref, (0.0, 1.0)).all()
        return got.shape == ref.shape and np.array_equal(got, ref)

    def actions(t):
        a = drive(None, n, t, eng.hero)
        if table is None:
            return a
        return np.argmin(((table[None] - a[:, None]) ** 2).sum(-1), axis=1).astype(np.int64)

    pin = None
    c = dict(compared=0, episodes=0, auto_resets=0, masked_resets=0, same_step_resets=0, mirror_resets=0,
             inside_repeat=0, reset_inside_repeat=0, unpinned=0, ring_slots=eng.L)
    causes = {}
    pool = OraclePool(n, scenes, oracle_args(row), size=size)
    try:
        ref = pool.run([("reset", i % S) for i in range(n)])
        obs = observe()
        for i in range(n):
            assert same_obs(obs[i], ref[i]["obs"]), (i, "reset observation")
        done = np.zeros(n, bool)
        unpinned = np.zeros(n, bool)  # test_gpu_scale's RETREAT NOTE: followed, not compared, until the next reset
        episodes = np.zeros(n, dtype=np.int64)
        since_reset = np.zeros(n, dtype=np.int64)
        term_total = 0
        rows = []
        for t in range(steps):
            a = actions(t)
            if same_step:  # rows of envs that do not end in this call must keep their contents
                final_before = eng.final_obs.cpu().numpy().view(np.uint8)
            if host:  # vector_env.py: pinned host actions, host mirrors of reward / flags / episode rows
                if pin is None:
                    pin = torch.from_numpy(np.zeros_like(a)).pin_memory()
                pin.numpy()[...] = a
                eng.step_host_full(pin, episode=True)
            else:
                eng.step(torch.from_numpy(a).cuda())
            head = eng.head
            cmds = []
            for i in range(n):
                if done[i]:
                    cmds.append(("reset", int(autoreset_scene(seed, i, int(episodes[i]), S))))
                else:
                    cmds.append(("repeat", (a[i], K)) if K > 1 else ("step", a[i]))
            ref = pool.run(cmds)
            rew = eng.reward.cpu().numpy()
            term = eng.terminated.cpu().numpy().astype(bool)
            trunc = eng.truncated.cpu().numpy().astype(bool)
            cause = eng.cause.cpu().numpy()
            hero = eng.hero.cpu().numpy()
            episode = eng.episode.cpu().numpy()
            if host:
                eng.wait_host_outputs()
                assert np.array_equal(eng.host_reward.numpy().view(np.int64), rew.view(np.int64)), (t, "host reward")
                assert np.array_equal(eng.host_terminated.numpy().astype(bool), term), (t, "host terminated")
                assert np.array_equal(eng.host_truncated.numpy().astype(bool), trunc), (t, "host truncated")
                assert np.array_equal(eng.host_episode.numpy()[term], episode[term]), (t, "host episode rows")
            term_total += int(term.sum())
            obs = observe()
            act = eng.get_state(amax)[1]
            ended = term | trunc
            final = {}
            if same_step:
                got = eng.final_obs.cpu().numpy()
                assert np.array_equal(got.view(np.uint8)[~ended], final_before[~ended]), \
                    (t, "final_obs rows of envs that did not end changed", np.flatnonzero(~ended))
                if ended.any():
                    idx = np.flatnonzero(ended)
                    fin = eng.final_obs[torch.from_numpy(idx).cuda()]
                    final = dict(zip(idx, (eng.fuse_windows(fuse, fin) if fuse else fin).cpu().numpy()))
            for i in range(n):
                r = ref[i]
                if done[i]:  # NEXT_STEP: this call resets, ignores the action, reward 0, not terminated
                    assert np.array_equal(hero[i], r["hero"]), (t, i, "auto-reset hero block", hero[i], r["hero"])
                    assert rew[i] == 0.0 and not term[i] and not trunc[i] and cause[i] == 0, (t, i)
                    assert same_obs(obs[i], r["obs"]), (t, i, "auto-reset observation")
                    done[i] = unpinned[i] = False
                    since_reset[i] = 0
                    c["auto_resets"] += 1
                    c["mirror_resets"] += int(head >= mirror)
                    continue
                since_reset[i] += 1
                if unpinned[i]:
                    c["unpinned"] += 1
                    if term[i] or trunc[i]:  # follow the engine's episode boundary; both sides re-sync at the reset
                        if term[i]:
                            rows.append(episode[i][None])
                        done[i] = True
                        episodes[i] += 1
                    continue
                c["compared"] += 1
                # actor poses come from the exact tables until they run out (in simulator steps), then live stepping
                pose_tol = POSE_TOL if traj == 0 or since_reset[i] * K > traj else 1e-9
                assert abs(r["reward"] - rew[i]) < K * 1e-9, (t, i, "reward", r["reward"], rew[i])
                assert r["term"] == term[i] and r["trunc"] == trunc[i], (t, i, "flags", r["term"], r["trunc"])
                assert r["cause"] == cause[i], (t, i, "cause", r["cause"], cause[i])
                _check_hero(hero[i], r["hero"], pose_tol, (t, i))
                if same_step and ended[i]:  # the terminal window is in final_obs; obs and actors are the reset's
                    assert same_obs(final[i], r["obs"]), (t, i, "final_obs", int((final[i] != r["obs"]).sum()))
                else:
                    assert same_obs(obs[i], r["obs"]), (t, i, "observation", int((obs[i] != r["obs"]).sum()))
                na = len(r["actors"])
                if na and not (same_step and ended[i]):
                    assert np.allclose(act[i, :na, :4], r["actors"], rtol=POSE_TOL, atol=POSE_TOL), (t, i, "actor poses")
                    if np.any(act[i, :na, 7].astype(np.int64) & 32):
                        unpinned[i] = True  # a pedestrian has just switched to a retreat route
                if r["term"]:
                    _check_episode(episode[i], r["episode"], (t, i))
                    rows.append(r["episode"][None])
                if r["term"] or r["trunc"]:
                    done[i] = True
                    episodes[i] += 1
                    c["episodes"] += 1
                    causes[int(r["cause"])] = causes.get(int(r["cause"]), 0) + 1
                    if K > 1 and r["j"] < K:
                        c["inside_repeat"] += 1
                        c["reset_inside_repeat"] += int(same_step)  # checked below, in this call
                else:
                    assert K == 1 or r["j"] == K, (t, i, "an agent step that did not end took", r["j"], "sub-steps")
            if same_step and ended.any():  # SAME_STEP: every env that ended was reset in this call, at this head
                assert np.array_equal(done, ended), t
                idx = np.flatnonzero(ended)
                scene = {i: int(autoreset_scene(seed, int(i), int(episodes[i]), S)) for i in idx}
                ref = pool.run([("reset", scene[i]) if ended[i] else None for i in range(n)])
                drawn = eng.snapshot(idx).header()[:, 0].cpu().numpy()
                for k, i in enumerate(idx):
                    assert drawn[k] == scene[i], (t, i, "same-step scene", drawn[k], scene[i])
                    assert same_obs(obs[i], ref[i]["obs"]), (t, i, "same-step reset observation")
                    na = len(ref[i]["actors"])
                    if na:
                        assert np.allclose(act[i, :na, :4], ref[i]["actors"], rtol=POSE_TOL, atol=POSE_TOL), \
                            (t, i, "same-step reset actor poses")
                c["same_step_resets"] += len(idx)
                c["mirror_resets"] += len(idx) * int(head >= mirror)
                done[:] = unpinned[ended] = False
                since_reset[ended] = 0
            if not next_step and not same_step and done.any():  # SyncVectorEnv-style masked reset of every env that ended
                ids = (np.arange(n) + 7 * (t + 1)) % S
                obs_r = eng.reset(torch.from_numpy(ids.astype(np.int32)), torch.from_numpy(done)).cpu().numpy()
                if fuse:
                    obs_r = observe()
                ref = pool.run([("reset", int(ids[i])) if done[i] else None for i in range(n)])
                for i in np.flatnonzero(done):
                    assert same_obs(obs_r[i], ref[i]["obs"]), (t, i, "masked reset observation")
                c["masked_resets"] += int(done.sum())
                c["mirror_resets"] += int(done.sum()) * int(eng.head >= mirror)
                unpinned[done] = False
                since_reset[done] = 0
                done[:] = False
    finally:
        pool.close()
    stats = eng.read_stats().cpu().numpy()
    eng.close()
    assert stats[0] == term_total, "episode counter != number of terminal flags raised"
    assert stats[-1] == steps * n, "the step counter counts calls x N"
    want = _stats_from_rows(np.concatenate(rows) if rows else np.zeros((0, len(E.EPISODE_FIELDS))))
    counts = [0, 2] + list(range(4, 12))  # CBEV_S_EPISODES, the summed lengths (simulator steps), per-cause counters
    assert np.array_equal(stats[counts], want[counts]), ("statistics counts", stats[counts], want[counts])
    sums = [k for k in range(len(stats) - 1) if k not in counts]
    assert np.allclose(stats[sums], want[sums], rtol=1e-7, atol=1e-7), ("statistics sums", stats[sums], want[sums])
    assert c["unpinned"] <= 0.25 * steps * n, c
    c["causes"] = {E.CAUSE_NAMES[k]: v for k, v in sorted(causes.items())}
    return c


MIN_EPISODES = 4  # compared terminal episodes per row


@pytest.mark.gpu
@pytest.mark.timeout(600)
@pytest.mark.parametrize("i", range(len(ROWS)), ids=[f"row{i:02d}" for i in range(len(ROWS))])
def test_row_against_the_oracle(i):
    row = _row(i)
    c = run_row(row)
    print(f"row{i:02d} {row} {c}")
    assert c["episodes"] >= MIN_EPISODES, c
    if row["autoreset"] == "next_step":
        assert c["auto_resets"] >= 1, c
    elif row["autoreset"] == "same_step":
        assert c["same_step_resets"] >= MIN_EPISODES, c
    else:
        assert c["masked_resets"] >= 1, c
    if row["repeat"] > 1:
        assert c["inside_repeat"] >= 1, c
        if row["autoreset"] == "same_step":
            assert c["reset_inside_repeat"] >= 1, c
    if row["ring_slots"] is not None:  # the smallest ring: some reset frames land in the mirror zone
        assert c["mirror_resets"] >= 1, c


def same_step_slices(row):
    """(window bytes, slices, slice bytes) of `cbev_launch_same_step_reset` for the row: slices of at least 16 KB, at
    most 32, 16-byte multiples, the last one possibly short."""
    if row["obs"] == "rgb":
        win = row["size"] * row["size"] * 3
    else:
        h, w = OBS_SIZE[row["resize"]][row["size"]]
        ch = 1 if row["mask"] in (None, "binary") else int(row["mask"].split("-")[0])
        win = row["frame_stack"] * h * w * {"f32": 4 * ch, "u8": ch, "gray": 1}[row["obs"]]
    min_slice = 16 << 10
    slices = min(32, -(-win // min_slice))
    size = (-(-win // slices) + 15) & ~15
    return win, -(-win // size), size


def test_same_step_copy_slices_are_covered():
    """k_same_step_reset copies slice j of env e's terminal window from CTA (e + j) mod N.  The same-step rows meet one
    slice, more slices than envs (the CTA index wraps, and one CTA serves two slices of one env), the 32-slice cap
    (windows above 512 KB) and a short last slice."""
    cases = set()
    for i in range(len(ROWS)):
        r = _row(i)
        if r["autoreset"] != "same_step":
            continue
        win, slices, size = same_step_slices(r)
        assert 1 <= slices <= 32 and size % 16 == 0 and (slices - 1) * size < win <= slices * size, (r, win, size)
        if slices == 1:
            cases.add("one slice")
        if r["n_envs"] < slices:
            cases.add("more slices than envs")
        if slices == 32 and win > 32 * (16 << 10):
            cases.add("32-slice cap")
        if win % size:
            cases.add("short last slice")
    assert cases == {"one slice", "more slices than envs", "32-slice cap", "short last slice"}, cases
    # the arithmetic against hand-computed windows: 7-class float32 96 x 96, F = 4 (1,032,192 B, 32 x 32,256 B) and
    # gray 84 x 84, F = 3 (21,168 B: two slices of 10,592 B, the last one 16 bytes short)
    assert same_step_slices(dict(obs="f32", resize="fast96", size=128, mask="7-class", frame_stack=4)) == \
        (1032192, 32, 32256)
    assert same_step_slices(dict(obs="gray", resize="area", size=128, mask=None, frame_stack=3)) == (21168, 2, 10592)


def _axis_values(row):
    """A row's values on the axes (K > 1 counts as the repeat value 3)."""
    v = {ax: row[ax] for ax in AXES}
    v["repeat"] = 1 if row["repeat"] == 1 else 3
    return v


def test_rows_are_the_generator_output():
    assert [dict(zip(COLUMNS, r)) for r in ROWS] == generate()


def test_every_allowed_pair_appears_in_a_row():
    covered = set()
    for i in range(len(ROWS)):
        covered |= _pairs(_axis_values(_row(i)))
    missing = allowed_pairs() - covered
    assert not missing, sorted(missing, key=_key)[:20]
    # spot checks of the rules: pairs that no valid configuration has are not asked for
    assert ("size", 256, "resize", "enlarge") not in allowed_pairs()
    assert ("mask", "binary", "fusion", "vehicle_temporal") not in allowed_pairs()
    assert ("size", 64, "resize", "fast96") not in allowed_pairs()


def test_every_row_respects_the_constraints():
    shortcut_off = set()
    for i in range(len(ROWS)):
        r = _row(i)
        assert not _conflict(_axis_values(r)), r
        assert set(COLUMNS) == set(r) and all(r[ax] is not None for ax in AXES if ax not in OPTIONAL), r
        if r["fusion"] not in (None, "stack"):  # fusion: semantic masks with a vehicle channel, F >= 3
            assert r["obs"] in ("f32", "u8") and r["mask"] in VEHICLE_MASKS and r["frame_stack"] >= 3, r
        if r["obs"] == "rgb":  # raw RGB: F = 1, no fusion, no resize
            assert r["frame_stack"] is None and r["fusion"] is None and r["resize"] == "raw", r
        if r["obs"] == "u8":
            h, w = OBS_SIZE[r["resize"]][r["size"]]
            assert h * w % 16 == 0, r
        if r["resize"] == "fast96":
            assert r["size"] == 128, r
        if r["resize"] == "block83":
            h, w = OBS_SIZE["block83"][r["size"]]
            assert 3 * r["size"] == 8 * h == 8 * w, r
            if not r["fov"]:
                shortcut_off.add(r["size"])
        assert 12 <= r["n_envs"] <= 24 and 80 <= r["steps"] <= 120 and r["repeat"] in (1, 3, 4, 8), r
    assert shortcut_off == set(AXES["size"]), "every scale needs a row that takes the 8:3 shortcut (FOV mask off)"
    assert any(r[COLUMNS.index("n_envs")] % 16 for r in ROWS)
    assert {r[COLUMNS.index("repeat")] for r in ROWS} == {1, 3, 4, 8}


def test_every_row_passes_host_validation():
    """EnvConfig's validation, cbev_create's argument checks (rc != CBEV_ERR_ARG; without a GPU it then fails to
    allocate) and the action-repeat range of every row."""
    import ctypes

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.config import EnvConfig

    lib = E.load_library()
    for i in range(len(ROWS)):
        r = _row(i)
        o = oracle_args(r)
        EnvConfig(size=r["size"], obs_size=o["obs_size"],
                  obs_mode="bev_semantic" if r["obs"] in ("f32", "u8") else "bev_rgb",
                  semantic_mask_ch=o["semantic_mask_ch"], temporal_fusion_mode=o["temporal_fusion_mode"],
                  fov_masked=r["fov"], ego_anchor_x_frac=r["anchor"][0], ego_anchor_y_frac=r["anchor"][1],
                  frame_stack=o["frame_stack"], action_mode=o["action_mode"],
                  action_profile_id=o["action_profile"], reward_mode=r["reward"])
        kw = engine_args(r)
        E._check_repeat(r["repeat"])
        cfg = E.CbevConfig()
        cfg.num_envs, cfg.fov_size = r["n_envs"], kw["size"]
        cfg.anchor_x_frac, cfg.anchor_y_frac = kw["anchor"]
        cfg.obs_h, cfg.obs_w = kw["obs_size"]
        cfg.obs_mode = E.OBS_SEMANTIC_U8 if kw["mask_dtype"] == "uint8" else kw["obs_mode"]
        cfg.mask_mode = E.MASK_MODES[kw["mask_mode"]]
        cfg.frame_stack, cfg.ring_slots = kw["frame_stack"], kw["ring_slots"] or 2 * kw["frame_stack"]
        cfg.action_mode, cfg.n_discrete = kw["action_mode"], len(kw["discrete_table"] or ()) or 1
        cfg.reward_mode, cfg.autoreset, cfg.max_actors = kw["reward_mode"], kw["autoreset"], 16
        cfg.trajectory_steps = kw["trajectory_steps"]
        h = ctypes.c_void_p()
        rc = lib.cbev_create(ctypes.byref(cfg), ctypes.byref(h))
        assert rc != 1, (i, r, lib.cbev_last_error().decode())
        if rc == 0:
            lib.cbev_destroy(h)

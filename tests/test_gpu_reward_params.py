"""Non-default reward parameters, batched engine vs oracle.

Every CaRL and shaping parameter of cbev_config reaches the kernels' reward code (judge_body, shared by the step, action
repeat and lookahead).  Goldens pin that code only at the defaults, so here each parameter set runs through
`run_scale_parity` with every env compared (sample = N): reward, flags, cause, the hero block, the episode rows and the
statistics vector against `OracleEnv` given the same parameters.  The values are distinct and not round, so two
swapped coefficients cannot give the same reward.

N = 83 is not a multiple of the envs per CTA (16 with G = 8, 4 with G = 32).  The narrow group path (G = 8) runs
with trajectory tables on; the wide one (G = 32) with more than 8 actor slots and `trajectory_steps=0`.  The pool
mixes rdm scenes with 16 vehicles (TTC), lead_brake and jaywalk.  Envs drive by index: route pursuit at cruise speed,
full throttle past the 35 km/h limit, a steady lateral bias onto the sidewalks, and hard braking after a run-up
(which ends in reverse).  The oracle counts the env-steps on which each parameter's term was active
(`oracle_pool.active_terms`); each set asserts a minimum for the terms it changes, so that no set passes without
reaching them."""
import numpy as np
import pytest

from golden_util import load_map
from test_gpu_scale import run_scale_parity

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

N_ENVS = 83
MIN_ACTIVE = 20  # env-steps on which a term under test must have been active


def _carl_random():
    r = np.random.default_rng(20261021)
    return dict(lane_center_exponent=r.uniform(0.5, 2.5), lane_center_floor=r.uniform(0.05, 0.45),
                off_lane_penalty=r.uniform(0.02, 0.6), speed_penalty_scale=r.uniform(0.3, 0.9),
                speed_penalty_floor=r.uniform(0.05, 0.45), ttc_threshold=r.uniform(2.5, 8.0),
                ttc_penalty_floor=r.uniform(0.55, 0.9))


def _shaping_random():
    """Every k_* (and the other coefficients) scaled by its own random factor away from the default."""
    from carlabev_env_b200.config import SHAPING_DEFAULTS

    r = np.random.default_rng(5021)
    p = {k: v * r.uniform(0.4, 2.5) for k, v in SHAPING_DEFAULTS.items() if isinstance(v, float)}
    p.update(offroad_terminate_after=4, max_actions=5000)
    return p


# (reward mode, parameters, terms that must be active, terms that must never be active)
SETS = {
    # carl_safety_v1 without reward_scale / comfort_penalty_floor, which the engine rejects (not implemented)
    "carl_safety": ("carl", dict(lane_center_exponent=1.5, lane_center_floor=0.15, off_lane_penalty=0.05,
                                 speed_penalty_scale=4.0, speed_penalty_floor=0.05, ttc_threshold=5.0,
                                 ttc_penalty_floor=0.05),
                    ("lane", "lane_floor", "off_lane", "speeding", "ttc"), ()),
    "carl_random": ("carl", _carl_random(), ("lane", "lane_floor", "off_lane", "speeding", "speed_floor", "ttc"), ()),
    "shaping_random": ("shaping", _shaping_random(),
                       ("sidewalk", "offroad_term", "route_dev", "align", "flow_cap", "reverse"), ("truncation",)),
    "shaping_offroad_off": ("shaping", dict(offroad_terminate_after=0, sidewalk_step_penalty=-0.0713,
                                            sidewalk_penalty_scale=-0.00917),
                            ("sidewalk",), ("offroad_term",)),
    "shaping_offroad_2": ("shaping", dict(offroad_terminate_after=2, sidewalk_step_penalty=-0.1531,
                                          sidewalk_penalty_scale=-0.0237),
                          ("sidewalk", "offroad_term"), ()),
    "shaping_small_bars": ("shaping", dict(route_dev_start=1.37, k_route_dev=0.0173, lat_clip=0.611,
                                           k_lat_quadratic=0.0291, lat_small=0.433, yaw_small=0.291,
                                           k_align_bonus=0.0347, max_speed_for_flow=3.17),
                           ("route_dev", "lat_clip", "align", "flow_cap"), ()),
    "shaping_max_actions": ("shaping", dict(max_actions=37, k_progress=0.0817, k_flow=0.0163),
                            ("truncation", "flow_cap"), ()),
}

# (parameter set, wide group path, auto-reset at the next step): every set once, both paths and both reset modes
CASES = [("carl_safety", False, True), ("carl_random", True, False), ("shaping_random", True, True),
         ("shaping_offroad_off", False, False), ("shaping_offroad_2", False, True),
         ("shaping_small_bars", True, False), ("shaping_max_actions", False, True)]


def _scenes():
    from carlabev_env_b200.pool import load_shipped_pool
    from carlabev_env_b200.scenes import build_scripted_scene

    cls = load_map()
    rdm = load_shipped_pool("rdm_rt_medium_v1")
    out = list(rdm[:12])
    out += [build_scripted_scene("lead_brake", 4100 + i, level=1 + i % 3, cls_map=cls) for i in range(6)]
    out += [build_scripted_scene("jaywalk", 4200 + i, level=1 + i % 4, cls_map=cls) for i in range(6)]
    return out


def drive(rng, n, t, hero):
    """Continuous actions by env index from the engine's last hero block: i % 4 == 0 pursues the route at cruise
    speed, 1 at full throttle, 2 with a steady lateral bias (left or right by i // 4), 3 brakes hard after a 2 s run-up.
    A hero block of a fresh episode (t == 0) has no set point: steer straight."""
    from carlabev_env_b200 import engine as E

    h = hero.cpu().numpy()
    H = {k: c for c, k in enumerate(E.HERO_FIELDS)}
    x, y, yaw, v = h[:, H["x"]], h[:, H["y"]], h[:, H["yaw"]], h[:, H["v"]]
    sx, sy, syaw = h[:, H["set_point_x"]], h[:, H["set_point_y"]], h[:, H["set_point_yaw"]]
    wrap = lambda a: (a + np.pi) % (2 * np.pi) - np.pi  # noqa: E731
    lat = -(x - sx) * np.sin(syaw) + (y - sy) * np.cos(syaw)  # > 0: left of the route
    steer = np.clip(1.2 * wrap(syaw - yaw) - 0.25 * lat, -1.0, 1.0)
    steer[h[:, H["t"]] == 0.0] = 0.0
    i = np.arange(n)
    kind = i % 4
    gas = np.where(v < 20.0, 0.6, 0.0)
    brake = np.where(v > 28.0, 0.3, 0.0)
    gas[kind == 1], brake[kind == 1] = 1.0, 0.0
    bias = np.where((i // 4) % 2 == 0, 0.3, -0.3)
    steer = np.where(kind == 2, np.clip(steer + bias, -1.0, 1.0), steer)
    gas = np.where(kind == 2, np.where(v < 15.0, 0.5, 0.0), gas)
    late = h[:, H["t"]] >= 2.0
    gas = np.where(kind == 3, np.where(late, 0.0, 1.0), gas)
    brake = np.where(kind == 3, np.where(late, 1.0, 0.0), brake)
    return np.stack([gas, steer, brake], axis=1).astype(np.float32)


@pytest.mark.parametrize("name,wide,next_step", CASES)
def test_reward_parameters_against_the_oracle(name, wide, next_step):
    from carlabev_env_b200 import engine as E

    mode, params, active, never = SETS[name]
    engine_kw = dict(action_mode=E.ACTION_CONTINUOUS, reward_params=params,
                     reward_mode=E.REWARD_CARL if mode == "carl" else E.REWARD_SHAPING,
                     autoreset=E.AUTORESET_NEXT_STEP if next_step else E.AUTORESET_DISABLED,
                     trajectory_steps=0 if wide else 1024)
    oracle_kw = dict(action_mode="continuous", reward_mode=mode, reward_params=params)
    n_auto, n_term, terms = run_scale_parity(_scenes(), N_ENVS, steps=150, make_actions=drive, engine_kw=engine_kw,
                                             oracle_kw=oracle_kw, sample=N_ENVS, seed=29,
                                             min_autoresets=1 if next_step else 0)
    print(f"coverage {name} wide={wide} next_step={next_step} episodes={n_term} auto_resets={n_auto} {terms}")
    low = {k: terms.get(k, 0) for k in active if terms.get(k, 0) < MIN_ACTIVE}
    assert not low, (name, "terms active on too few env-steps", low, terms)
    seen = {k: terms[k] for k in never if terms.get(k, 0)}
    assert not seen, (name, "terms that this set switches off were active", seen)
    assert n_term >= 20, n_term


def test_engine_rejects_unknown_and_unimplemented_reward_parameters():
    from carlabev_env_b200 import engine as E

    with pytest.raises(E.CbevError, match="unknown reward parameter 'k_progres'"):
        E.Engine(1, action_mode=E.ACTION_CONTINUOUS, reward_params=dict(k_progres=0.1), ring_budget_bytes=1 << 20)
    for k in ("zero_speed_reward_offroad", "zero_progress_reward_offroad"):
        with pytest.raises(E.CbevError, match=f"reward parameter {k}=False is not implemented"):
            E.Engine(1, action_mode=E.ACTION_CONTINUOUS, reward_params={k: False}, ring_budget_bytes=1 << 20)

"""Oracle: per-step simulation (dynamics, scripted actors, collision, reward, stats).

TEST INFRASTRUCTURE ONLY -- see oracle/__init__.py.  Plain Python/NumPy restatement
of the reference's per-env step.  Line references are into /root/reference/CarlaBEV.

A *scene* is a dict of NumPy arrays (one entry of the scene pool, SURVEY.md App. B):
  ego_state0 f64[4] (x,y,yaw,v)  ego_target_speed f64  ego_tidx0 i32
  ego_cx/ego_cy/ego_cyaw f64[Pe] (smoothed route)      rew_rx/rew_ry i32[Pr] (raw route)
  route_length_m f64  len_ego_route f64  num_vehicles i32
  act_kind u8[A] (0 vehicle, 1 pedestrian)  act_state0 f64[A,4]  act_tidx0 i32[A]
  act_cruise_px/act_cruise_mps f64[A]  act_route_off i32[A+1]  act_cx/act_cy/act_cyaw f64[sum P]
  act_raw_off i32[A+1]  act_raw_x/act_raw_y f64[sum R] (authored route, used by the retreat FSM)
  act_beh u8[A]  act_beh_p f64[A,4]       tl_rect i32[L,4]  tl_color u8[L]
"""
from __future__ import annotations

import math

import numpy as np

# --- constants (SURVEY.md A.1) ---------------------------------------------------
DT = 0.1                      # stanley_controller.py:22, scene.py:30
WHEEL_BASE = 2.9              # stanley_controller.py:29 (used in pixel units)
K_STANLEY = 2.0               # stanley_controller.py:20
KP_SPEED = 1.0                # stanley_controller.py:21
MAX_STEER = np.radians(30.0)  # stanley_controller.py:28
MPP = 40.0 / 128.0            # hero.py:67, carl_reward_fn.py:15-16
LANE_HALF_WIDTH_M = 3.0       # carl_reward_fn.py:17
MIN_DIST = 35                 # carlabev.py:173
SPEED_LIMIT = 35              # scene.py:215

KIND_VEHICLE, KIND_PEDESTRIAN = 0, 1
BEH_NONE, BEH_LEAD_BRAKE, BEH_CROSS, BEH_STOP_MID, BEH_STOP_RETURN = 0, 1, 2, 3, 4
# jaywalk FSM states (behavior/jaywalk.py)
(ST_IDLE, ST_WAITING, ST_ENTERING, ST_YIELDING, ST_CROSSING, ST_STALLED,
 ST_RETREATING, ST_CLEARED, ST_RETREATED) = range(9)

# collision result codes (scene.py:110-140)
HIT_NONE, HIT_VEHICLE, HIT_PEDESTRIAN, HIT_TARGET = 0, 1, 2, 3
# termination causes (carlabev.py:43-49 + "ckpt")
CAUSE_NONE, CAUSE_CKPT, CAUSE_COLLISION, CAUSE_SUCCESS, CAUSE_OOB, CAUSE_OFFROAD, CAUSE_MAX_ACTIONS, CAUSE_UNKNOWN = range(8)
CAUSE_NAMES = (None, "ckpt", "collision", "success", "out_of_bounds", "off_road", "max_actions", "unknown")
TERMINAL_CAUSES = (CAUSE_COLLISION, CAUSE_SUCCESS, CAUSE_OOB, CAUSE_OFFROAD, CAUSE_MAX_ACTIONS)

# map classes (semantics.py:8-17, 34-38)
CLS_NON_DRIVABLE, CLS_DRIVABLE, CLS_SIDEWALK = 0, 1, 2

COMFORT_KEYS = ("accel_long", "accel_lat", "jerk_long", "jerk_lat", "yaw_rate", "yaw_acc")
COMFORT_BOUNDS = {"accel_long": 2.0, "accel_lat": 2.0, "yaw_rate": 20.0,
                  "jerk_long": 3.0, "jerk_lat": 3.0, "yaw_acc": 120.0}  # comfort.py:3-10

DISCRETE9 = ((0, 0, 0), (1, 0, 0), (0, 0, 1), (1, 1, 0), (1, -1, 0), (0, 1, 0), (0, -1, 0), (0, 1, 1), (0, -1, 1))
DISCRETE13 = ((0, 0, 0), (1, 0, 0), (0, 0, 1), (1, 1, 0), (1, .5, 0), (1, -.5, 0), (1, -1, 0), (0, 1, 0),
              (0, .5, 0), (0, -.5, 0), (0, -1, 0), (0, 1, 1), (0, -1, 1))  # action_profiles.py:35-76


def angle_mod(x):
    """control/utils.py:29-86 default branch ([-pi, pi), NumPy floor-mod)."""
    return ((np.asarray(x).flatten() + np.pi) % (2 * np.pi) - np.pi).item()


def smooth_route(ax, ay, window=11, poly=3):
    """control/utils.py:200-269 (cx, cy, cyaw only)."""
    from scipy.signal import savgol_filter

    ax = np.asarray(ax, dtype=float)
    ay = np.asarray(ay, dtype=float)
    d = np.hypot(np.diff(ax), np.diff(ay))
    keep = np.concatenate(([True], d > 1e-9))
    ax, ay = ax[keep], ay[keep]
    if len(ax) < 2:
        ax = np.array([ax[0], ax[0] + 1e-3])
        ay = np.array([ay[0], ay[0]])
    if window % 2 == 0:
        window += 1
    if window > len(ax):
        window = len(ax) if len(ax) % 2 == 1 else len(ax) - 1
    if window < 3:
        window = 3
    poly = min(poly, window - 1)
    if len(ax) >= window:
        cx = savgol_filter(ax, window_length=window, polyorder=poly)
        cy = savgol_filter(ay, window_length=window, polyorder=poly)
    else:
        cx, cy = ax.copy(), ay.copy()
    s = np.concatenate(([0.0], np.cumsum(np.hypot(np.diff(cx), np.diff(cy)))))
    if s[-1] <= 1e-9:
        return cx, cy, np.zeros_like(cx)
    cyaw = np.unwrap(np.arctan2(np.gradient(cy, s), np.gradient(cx, s)))
    return cx, cy, cyaw


class Body:
    """State + Controller (control/state.py, control/stanley_controller.py)."""

    __slots__ = ("x", "y", "yaw", "v", "x_1", "y_1", "yaw_1", "v_1", "target", "tidx", "cx", "cy", "cyaw")

    def nearest(self):
        """calc_target_index, stanley_controller.py:100-123."""
        fx = self.x + WHEEL_BASE * np.cos(self.yaw)
        fy = self.y + WHEEL_BASE * np.sin(self.yaw)
        dx = fx - self.cx
        dy = fy - self.cy
        idx = int(np.argmin(np.hypot(dx, dy)))
        vec = [-np.cos(self.yaw + np.pi / 2), -np.sin(self.yaw + np.pi / 2)]
        err = np.dot([dx[idx], dy[idx]], vec)
        return idx, err

    def stanley(self):
        """stanley_control, stanley_controller.py:64-89."""
        idx, err = self.nearest()
        if self.tidx >= idx:
            idx = self.tidx
        theta_e = angle_mod(self.cyaw[idx] - self.yaw)
        theta_d = np.arctan2(K_STANLEY * err, max(self.v, 1e-3))
        delta = np.clip(theta_e + theta_d, -MAX_STEER, MAX_STEER)
        return delta, idx

    def update(self, acc, delta):
        """State.update, state.py:29-51."""
        delta = np.clip(delta, -MAX_STEER, MAX_STEER)
        self.x_1, self.y_1, self.yaw_1, self.v_1 = self.x, self.y, self.yaw, self.v
        self.x += self.v * np.cos(self.yaw) * DT
        self.y += self.v * np.sin(self.yaw) * DT
        self.yaw += self.v / WHEEL_BASE * np.tan(delta) * DT
        self.v += acc * DT
        self.yaw = angle_mod(self.yaw)
        self.v = np.clip(self.v, -1 * self.target, self.target)

    def control_step(self):
        """Controller.control_step, stanley_controller.py:51-62 (freeze at route end)."""
        if self.tidx >= len(self.cx) - 1:
            self.target = 0.0
            return
        ai = KP_SPEED * (self.target - self.v)
        di, self.tidx = self.stanley()
        self.update(ai, di)

    def set_route(self, ax, ay, v0):
        """Controller.set_route with jitter_start=False (mid-episode retreat),
        stanley_controller.py:34-49."""
        self.cx, self.cy, self.cyaw = smooth_route(ax, ay, window=11, poly=3)
        self.x, self.y = self.cx[0], self.cy[0]
        self.v = v0
        self.tidx, _ = self.nearest()
        self.yaw = self.cyaw[self.tidx]


class Actor(Body):
    __slots__ = ("kind", "size", "cruise_px", "cruise_mps", "target_speed", "target_mps", "beh", "p",
                 "raw_x", "raw_y", "rx_len", "fsm", "elapsed", "state_elapsed", "braking", "retreat_goal")

    # actor.py:121-133
    def set_target_mps(self, mps):
        mps = max(0.0, float(mps))
        self.target_mps = mps
        self.target_speed = float(mps) / MPP

    def _set_state(self, st, mps=None):
        self.fsm = st
        self.state_elapsed = 0.0
        if mps is not None:
            self.set_target_mps(mps)

    def _mid_idx(self):  # jaywalk.py:34-35
        return max(1, min(self.rx_len - 1, int(self.p[1] * (self.rx_len - 1))))

    def _complete(self):  # jaywalk.py:37-38
        return self.tidx >= self.rx_len - 1

    def _start_retreat(self):  # jaywalk.py:43-54
        cur = max(0, min(self.tidx, self.rx_len - 1))
        rrx = [self.x] + list(self.raw_x[: cur + 1][::-1])
        rry = [self.y] + list(self.raw_y[: cur + 1][::-1])
        self.retreat_goal = np.array([self.raw_x[0], self.raw_y[0]], dtype=float)
        self.rx_len = len(rrx)
        self.set_route(rrx, rry, self.v)
        self._set_state(ST_RETREATING, self.cruise_mps)

    def apply_behavior(self, t, dt):
        b = self.beh
        if b == BEH_NONE:
            return
        if b == BEH_LEAD_BRAKE:  # lead_brake.py:10-15
            if t >= self.p[0]:
                self.braking = True
            if self.braking:
                self.set_target_mps(self.target_mps - self.p[1] * dt)
            return
        # jaywalk family (jaywalk.py:56-138); p = (start_delay, trigger_fraction, stop_duration|-1, retreat)
        self.elapsed += dt
        self.state_elapsed += dt
        st = self.fsm
        cruise = self.cruise_mps
        if b == BEH_CROSS:  # jaywalk.py:114-138
            if st == ST_WAITING:
                self.set_target_mps(0.0)
                if self.elapsed >= self.p[0]:
                    self._set_state(ST_CROSSING, cruise)
            elif st == ST_CROSSING:
                self.set_target_mps(cruise)
                if self._complete():
                    self._set_state(ST_CLEARED, 0.0)
            elif st == ST_CLEARED:
                self.set_target_mps(0.0)
            return
        stop_duration = None if self.p[2] < 0 else self.p[2]
        retreat = self.p[3] != 0
        if st == ST_WAITING:
            self.set_target_mps(0.0)
            if self.elapsed >= self.p[0]:
                self._set_state(ST_ENTERING, cruise)
        elif st == ST_ENTERING:
            self.set_target_mps(cruise)
            if self.tidx >= self._mid_idx():
                if retreat:
                    self._set_state(ST_YIELDING, 0.0)
                elif stop_duration is None:
                    self._set_state(ST_STALLED, 0.0)
                else:
                    self._set_state(ST_YIELDING, 0.0)
            elif self._complete():
                self._set_state(ST_CLEARED, 0.0)
        elif st == ST_YIELDING:
            self.set_target_mps(0.0)
            if stop_duration is None:
                return
            if self.state_elapsed >= stop_duration:
                if retreat:
                    self._start_retreat()
                else:
                    self._set_state(ST_CROSSING, cruise)
        elif st == ST_CROSSING:
            self.set_target_mps(cruise)
            if self._complete():
                self._set_state(ST_CLEARED, 0.0)
        elif st == ST_STALLED:
            self.set_target_mps(0.0)
        elif st == ST_RETREATING:
            self.set_target_mps(cruise)
            reached = False
            if self.retreat_goal is not None:
                reached = np.linalg.norm(np.array([self.x, self.y], dtype=float) - self.retreat_goal) <= 1.0
            if reached or self._complete():
                self._set_state(ST_RETREATED, 0.0)
        elif st in (ST_CLEARED, ST_RETREATED):
            self.set_target_mps(0.0)

    def step(self, t, dt):
        """Actor.step, actor.py:110-119."""
        self.apply_behavior(t, dt)
        self.target = self.target_speed
        self.control_step()


def rect_left(center_world, pad, size):
    """SurfaceFrame.rect_from_world_center + Rect.center setter (transforms.py:46-51):
    Python banker's round of (pad + coord), then left = centre - size//2."""
    return round(float(pad) + float(center_world) * 1.0) - (size >> 1)


def rects_overlap(ax, ay, aw, bx, by, bw):
    """pygame Rect.colliderect for positive square sizes (strict half-open overlap)."""
    return ax < bx + bw and ay < by + bw and ax + aw > bx and ay + aw > by


class SceneSim:
    """One environment's world: ego + scripted actors + targets (scene.py, actor_manager.py, hero.py)."""

    def __init__(self, scene, cls_map, pad, reward_mode="carl", reward_params=None, size=128):
        self.scene = scene
        self.scale = int(1024 / int(size))   # hero.py:14 (EnvConfig.size: 8 at the 128 scale)
        self.hero_w = int(32 / self.scale)   # hero.py:17: the ego square, 4 px at the 128 scale
        self.cls_map = cls_map  # (H, W) uint8 classes
        self.pad = int(pad)
        self.reward_mode = reward_mode
        self.rp = dict(reward_params or {})
        self.reset()

    # ------------------------------------------------------------------ reset
    def reset(self):
        s = self.scene
        e = Body()
        e.x, e.y, e.yaw, e.v = (s["ego_state0"][0], s["ego_state0"][1], s["ego_state0"][2], s["ego_state0"][3])
        e.x_1, e.y_1, e.yaw_1, e.v_1 = e.x, e.y, e.yaw, e.v
        e.target = float(s["ego_target_speed"])
        e.tidx = int(s["ego_tidx0"])
        e.cx, e.cy, e.cyaw = s["ego_cx"], s["ego_cy"], s["ego_cyaw"]
        self.ego = e
        self.acc = 0.0
        self.prev_comfort = None  # (accel_long, accel_lat, yaw_rate_deg)
        self.control = dict(cmd_gas=0.0, cmd_steer=0.0, cmd_brake=0.0, applied_delta=0.0)
        self.comfort = dict(speed_mps=0.0, accel_long=0.0, accel_lat=0.0, jerk_long=0.0, jerk_lat=0.0,
                            yaw_rate=0.0, yaw_acc=0.0)
        self.actors = []
        for i in range(len(s["act_kind"])):
            a = Actor()
            a.kind = int(s["act_kind"][i])
            a.size = 4 if a.kind == KIND_VEHICLE else 2  # vehicle.py:24, pedestrian.py:24
            a.x, a.y, a.yaw, a.v = (s["act_state0"][i, 0], s["act_state0"][i, 1], s["act_state0"][i, 2],
                                    float(s["act_state0"][i, 3]))
            a.x_1, a.y_1, a.yaw_1, a.v_1 = a.x, a.y, a.yaw, a.v
            a.tidx = int(s["act_tidx0"][i])
            lo, hi = int(s["act_route_off"][i]), int(s["act_route_off"][i + 1])
            a.cx, a.cy, a.cyaw = s["act_cx"][lo:hi], s["act_cy"][lo:hi], s["act_cyaw"][lo:hi]
            lo, hi = int(s["act_raw_off"][i]), int(s["act_raw_off"][i + 1])
            a.raw_x, a.raw_y = s["act_raw_x"][lo:hi], s["act_raw_y"][lo:hi]
            a.rx_len = hi - lo
            a.cruise_px = float(s["act_cruise_px"][i])
            a.cruise_mps = float(s["act_cruise_mps"][i])
            a.target_speed, a.target_mps = a.cruise_px, a.cruise_mps  # actor.py:94-95
            a.target = a.target_speed
            a.beh = int(s["act_beh"][i])
            a.p = [float(v) for v in s["act_beh_p"][i]]
            a.fsm, a.elapsed, a.state_elapsed, a.braking, a.retreat_goal = ST_IDLE, 0.0, 0.0, False, None
            if a.beh in (BEH_CROSS, BEH_STOP_MID, BEH_STOP_RETURN):  # jaywalk.py:23-28
                a.fsm = ST_WAITING
                a.set_target_mps(0.0)
            self.actors.append(a)
        # targets: one per smoothed ego route point (scenes/utils.py:114-122)
        self.tgt_x = np.asarray(e.cx, dtype=float)
        self.tgt_y = np.asarray(e.cy, dtype=float)
        self.tgt_visible = np.ones(len(self.tgt_x), dtype=bool)
        self.tgt_visible_at_draw = self.tgt_visible.copy()
        self.t = 0.0
        goal = np.array([self.tgt_x[-1], self.tgt_y[-1]])
        self.dist2goal = float(np.linalg.norm(np.array([e.x, e.y], dtype=float) - goal))
        self.dist2goal_1 = self.dist2goal
        # reward state
        self.rew_route = list(zip(s["rew_rx"], s["rew_ry"]))
        self.rew_len = [0.0]
        for i in range(1, len(self.rew_route)):  # carl_reward_fn.py:20-26
            dx = self.rew_route[i][0] - self.rew_route[i - 1][0]
            dy = self.rew_route[i][1] - self.rew_route[i - 1][1]
            self.rew_len.append(self.rew_len[-1] + np.hypot(dx, dy))
        self.s_prev = None
        self.k = 0
        self.consecutive_offroad = 0
        self.last_delta_yaw = 0.0
        self.stats_reset()

    # -------------------------------------------------------------- dynamics
    def ego_step(self, gas, steer, brake):
        """BaseAgent.physics_step, hero.py:88-138 (dtype ledger SURVEY.md A.2)."""
        e = self.ego
        _, e.tidx = e.stanley()
        f32 = np.float32
        acc_val = float(f32(gas) * f32(self.scale)) if gas > 0 else 0.0          # hero.py:140-142
        if abs(e.v) < 0.1:                                                  # hero.py:144-158
            delta = 0.0
        else:
            steer_deg = np.clip(18.0 / (1.0 + 0.35 * abs(e.v)), 8.0, 18.0)
            delta = math.radians(float(f32(steer)) * steer_deg)
        speed_factor = np.clip(abs(e.v) / 5.0, 0.3, 1.0)                    # hero.py:160-162
        brake_val = (float((f32(brake) * f32(0.6)) * f32(self.scale)) if brake > 0 else 0.0) * speed_factor
        target_acc = acc_val - brake_val - 0.05 * e.v
        alpha = 0.2
        self.acc = (1 - alpha) * self.acc + alpha * target_acc
        e.update(self.acc, delta)
        e.v *= 0.9999
        if abs(e.v) < 0.05:
            e.v = 0.0
        e.v *= 0.985
        self.control = dict(cmd_gas=float(gas), cmd_steer=float(steer), cmd_brake=float(brake),
                            applied_delta=float(delta))
        # compute_comfort_kinematics, comfort.py:17-61
        speed_mps = float(e.v) * MPP
        prev_speed_mps = float(e.v_1) * MPP
        dyaw = float(e.yaw) - float(e.yaw_1)
        yaw_rate_rad = math.atan2(math.sin(dyaw), math.cos(dyaw)) / DT
        yaw_rate_deg = math.degrees(yaw_rate_rad)
        accel_long = (speed_mps - prev_speed_mps) / DT
        accel_lat = speed_mps * yaw_rate_rad
        if self.prev_comfort is None:
            jerk_long = jerk_lat = yaw_acc = 0.0
        else:
            jerk_long = (accel_long - float(self.prev_comfort[0])) / DT
            jerk_lat = (accel_lat - float(self.prev_comfort[1])) / DT
            yaw_acc = (yaw_rate_deg - float(self.prev_comfort[2])) / DT
        self.comfort = dict(speed_mps=speed_mps, accel_long=accel_long, accel_lat=accel_lat, jerk_long=jerk_long,
                            jerk_lat=jerk_lat, yaw_rate=yaw_rate_deg, yaw_acc=yaw_acc)
        self.prev_comfort = (accel_long, accel_lat, yaw_rate_deg)

    def decode_action(self, action, action_mode, table=DISCRETE9):
        """spaces.py:43-47 + hero.py:165-187."""
        if action_mode == "discrete":
            a = np.asarray(table[int(action)], dtype=np.float32)
            return a[0], a[1], a[2]
        a = np.asarray(action, dtype=np.float32)
        return np.clip(a[0], 0.0, 1.0), np.clip(a[1], -1.0, 1.0), np.clip(a[2], 0.0, 1.0)

    def scene_step(self, gas, steer, brake):
        """Scene._scene_step minus drawing, scene.py:90-105."""
        self.t += DT
        self.ego_step(gas, steer, brake)
        for a in self.actors:
            a.step(self.t, DT)
        # draw_all runs here, BEFORE collision_check consumes targets (scene.py:94-95)
        self.tgt_visible_at_draw = self.tgt_visible.copy()
        self.dist2goal_1 = self.dist2goal
        goal = np.array([self.tgt_x[-1], self.tgt_y[-1]])
        self.dist2goal = float(np.linalg.norm(np.array([self.ego.x, self.ego.y], dtype=float) - goal))

    # ------------------------------------------------------------- collision
    def tile_class(self):
        """BaseMap.semantic_tile_at, world.py:159-165."""
        h, w = self.cls_map.shape
        x = int(np.clip(round(float(self.ego.x)), 0, w - 1))
        y = int(np.clip(round(float(self.ego.y)), 0, h - 1))
        return int(self.cls_map[y, x])

    def hero_info(self):
        """Controller.controller_info, stanley_controller.py:163-176."""
        e = self.ego
        t = e.tidx
        sp = np.array([e.cx[t], e.cy[t], e.cyaw[t]])
        pos = np.array([float(e.x), float(e.y)])
        d = pos - sp[:-1]
        dist2wp = np.sqrt(d.dot(d))
        n = 5
        if t + n <= len(e.cx):
            wx, wy = e.cx[t:t + n], e.cy[t:t + n]
        else:
            wx, wy = e.cx[t:-1], e.cy[t:-1]
        return dict(state=[e.x, e.y, e.yaw, e.v], last_state=[e.x_1, e.y_1, e.yaw_1, e.v_1], dist2wp=dist2wp,
                    set_point=sp, next_wps=(wx, wy))

    def collision_check(self):
        """Scene.collision_check, scene.py:110-140: (hit, hit_id, nearby, tile_class)."""
        pad = self.pad
        e = self.ego
        hw = self.hero_w
        hx, hy = rect_left(e.x, pad, hw), rect_left(e.y, pad, hw)
        hcx, hcy = hx + (hw >> 1), hy + (hw >> 1)
        hit, hit_id = HIT_NONE, -1
        nearby = []
        for kind in (KIND_VEHICLE, KIND_PEDESTRIAN):  # dict order: vehicle, pedestrian (actor_manager.py:25-31)
            for a in self.actors:
                if a.kind != kind:
                    continue
                ax, ay = rect_left(a.x, pad, a.size), rect_left(a.y, pad, a.size)
                half = a.size >> 1
                dist = math.hypot(hcx - (ax + half), hcy - (ay + half))
                if abs(dist) < MIN_DIST:
                    nearby.append((a.x, a.y, a.v * np.cos(a.yaw), a.v * np.sin(a.yaw)))
                if rects_overlap(hx, hy, hw, ax, ay, a.size):
                    hit, hit_id = (HIT_VEHICLE if kind == KIND_VEHICLE else HIT_PEDESTRIAN), kind
        n = len(self.tgt_x)
        for i in range(n):  # target.py:37-44
            if not self.tgt_visible[i]:
                continue
            size = 4 if i == n - 1 else 2
            tx, ty = rect_left(self.tgt_x[i], pad, size), rect_left(self.tgt_y[i], pad, size)
            if rects_overlap(hx, hy, hw, tx, ty, size):
                self.tgt_visible[i] = False
                hit, hit_id = HIT_TARGET, i
        return hit, hit_id, nearby, self.tile_class()

    # ---------------------------------------------------------------- reward
    def _lateral_error(self, x, y, wx, wy):
        """control/utils.py:165-197 with signed=True."""
        min_error = float("inf")
        for i in range(len(wx) - 1):
            A = np.array([wx[i], wy[i]])
            B = np.array([wx[i + 1], wy[i + 1]])
            P = np.array([x, y])
            AB = B - A
            AP = P - A
            with np.errstate(all="ignore"):
                t = np.dot(AP, AB) / np.dot(AB, AB)
            t = np.clip(t, 0.0, 1.0)
            closest = A + t * AB
            dd = P - closest
            err = np.sqrt(dd.dot(dd))
            cross = AB[0] * AP[1] - AB[1] * AP[0]
            err *= np.sign(cross) if cross != 0 else 1
            if abs(err) < abs(min_error):
                min_error = err
        return min_error

    def _route_progress(self, px, py):
        """compute_route_progress, carl_reward_fn.py:29-58."""
        best_s, best_dist = 0, 1e9
        route, lengths = self.rew_route, self.rew_len
        for i in range(len(route) - 1):
            A = np.array(route[i])
            B = np.array(route[i + 1])
            P = np.array([px, py])
            AB = B - A
            t = np.dot(P - A, AB) / (np.dot(AB, AB) + 1e-9)
            t = np.clip(t, 0, 1)
            closest = A + t * AB
            dd = P - closest
            dist = np.sqrt(dd.dot(dd))
            if dist < best_dist:
                best_dist = dist
                ABf = AB.astype(float)
                best_s = lengths[i] + t * np.sqrt(ABf.dot(ABf))
        return best_s

    @staticmethod
    def _ttc_raw(hero_state, nearby, mpp):
        """compute_ttc_raw, reward_signals.py:45-94."""
        hx, hy, hyaw, hv = hero_state
        hx_m, hy_m = hx * mpp, hy * mpp
        hv_m = hv * mpp
        hvx, hvy = hv_m * np.cos(hyaw), hv_m * np.sin(hyaw)
        min_ttc = np.inf
        for ax, ay, avx, avy in nearby:
            rx, ry = ax * mpp - hx_m, ay * mpp - hy_m
            rvx, rvy = avx * mpp - hvx, avy * mpp - hvy
            r = np.array([rx, ry])
            norm = np.sqrt(r.dot(r))
            rel = (rvx * rx + rvy * ry) / (norm + 1e-6)
            if rel >= 0:
                continue
            min_ttc = min(min_ttc, abs(norm / rel))
        return min_ttc

    @staticmethod
    def _ttc_shaping(hero_state, nearby, thr):
        """compute_ttc, reward_signals.py:15-42."""
        hx, hy, hyaw, hv = hero_state
        hvx, hvy = hv * np.cos(hyaw), hv * np.sin(hyaw)
        min_ttc = np.inf
        for ax, ay, avx, avy in nearby:
            rx, ry = ax - hx, ay - hy
            rvx, rvy = avx - hvx, avy - hvy
            r = np.array([rx, ry])
            norm = np.sqrt(r.dot(r))
            rel = (rvx * rx + rvy * ry) / (norm + 1e-6)
            if rel >= 0:
                continue
            min_ttc = min(min_ttc, abs(norm / rel))
        if min_ttc < np.inf:
            return -np.exp(-min_ttc / thr)
        return 0.0

    def comfort_violations(self):
        """count_comfort_violations, comfort.py:64-70."""
        return sum(int(abs(float(self.comfort[k])) > float(lim)) for k, lim in COMFORT_BOUNDS.items())

    def carl_reward(self, hit, hit_id, nearby, tile, hero):
        """CaRLRewardFn.step, carl_reward_fn.py:149-341 -> (reward, terminated, cause)."""
        p = self.rp
        n_t = len(self.tgt_x)
        if tile == CLS_NON_DRIVABLE:
            return -1.0, True, CAUSE_COLLISION
        if hit == HIT_TARGET and hit_id == n_t - 1:
            return 1.0, True, CAUSE_SUCCESS
        if hit == HIT_TARGET:
            return 0.1, False, CAUSE_CKPT
        if hit in (HIT_VEHICLE, HIT_PEDESTRIAN):
            return -1.0, True, CAUSE_COLLISION
        if hero["dist2wp"] > 50:
            return -1.0, True, CAUSE_OOB
        x, y, yaw, speed = hero["state"]
        speed_mps = float(speed) * MPP
        s_t = self._route_progress(x, y)
        if self.s_prev is None:
            self.s_prev = s_t
        rc_raw = max(0.0, s_t - self.s_prev)
        self.s_prev = s_t
        total = self.rew_len[-1]
        rc = rc_raw / total if total > 0 else 0.0
        rc = float(np.clip(rc * 100, 0.0, 1.0))
        wx, wy = hero["next_wps"]
        d2r = self._lateral_error(x, y, wx, wy)
        dist_m = abs(d2r) * MPP
        if dist_m <= 0.0:
            p_route = 1.0
        else:
            p_route = max(p.get("lane_center_floor", 0.2),
                          1.0 - (dist_m / LANE_HALF_WIDTH_M) ** p.get("lane_center_exponent", 1.0))
        far = dist_m > (1.5 * LANE_HALF_WIDTH_M)
        off_lane = (tile == CLS_SIDEWALK) or far
        p_off = p.get("off_lane_penalty", 0.0) if off_lane else 1.0
        limit = float(SPEED_LIMIT)
        limit_mps = limit / 3.6 if limit > 20.0 else limit
        over = max(speed_mps - limit_mps, 0.0)
        if over <= 0.0:
            p_speed = 1.0
        else:
            p_speed = max(p.get("speed_penalty_floor", 0.1), float(np.exp(-over / p.get("speed_penalty_scale", 6.0))))
        ttc = self._ttc_raw(hero["state"], nearby, MPP)
        p_ttc = 0.5 if ttc < p.get("ttc_threshold", 4.0) else 1.0
        p_ttc = max(p.get("ttc_penalty_floor", 0.1), float(p_ttc))
        viol = self.comfort_violations()
        p_comfort = 1.0 - 0.5 * (viol / 6.0) if viol > 0 else 1.0
        P_t = 1.0
        for f in (float(p_route), p_off, p_speed, float(p_ttc), float(p_comfort)):
            P_t *= f
        reward = float(np.clip(rc * P_t, 0.0, 1.0))
        return reward, False, CAUSE_NONE

    def shaping_reward(self, hit, hit_id, nearby, tile, hero):
        """RewardFn.step/non_terminal/termination, reward.py:80-278."""
        p = self.rp
        g = p.get
        self.k += 1
        reward, terminated, cause = -0.002, False, CAUSE_NONE
        n_t = len(self.tgt_x)
        if self.k >= g("max_actions", 5000):
            return 0.0, True, CAUSE_MAX_ACTIONS
        if hero["dist2wp"] > 60:
            return -1.0, True, CAUSE_OOB
        if tile == CLS_NON_DRIVABLE:
            return -1.0, True, CAUSE_COLLISION
        if hit != HIT_NONE:
            if hit == HIT_PEDESTRIAN:
                return -20.0, True, CAUSE_COLLISION
            if hit == HIT_VEHICLE:
                return -12.0, True, CAUSE_COLLISION
            if hit_id == n_t - 1:
                return +18.0, True, CAUSE_SUCCESS
            return +0.7, False, CAUSE_CKPT
        on_sidewalk = tile == CLS_SIDEWALK
        if on_sidewalk:
            self.consecutive_offroad += 1
            reward += g("sidewalk_step_penalty", -0.12) + g("sidewalk_penalty_scale", -0.006) * self.consecutive_offroad
        else:
            self.consecutive_offroad = 0
        after = g("offroad_terminate_after", 40)
        if after and self.consecutive_offroad >= after:
            reward -= 0.7
            terminated, cause = True, CAUSE_OFFROAD
        else:
            reward += self._shaping_terms(nearby, hero, on_sidewalk)
        return float(np.clip(reward, -1.0, 1.0)), terminated, cause

    def _shaping_terms(self, nearby, hero, offroad):
        g = self.rp.get
        r = 0.0
        x, y, yaw, v = hero["state"]
        _, _, yaw_1, v_1 = hero["last_state"]
        desired_yaw = hero["set_point"][2]
        yaw_error = np.arctan2(np.sin(desired_yaw - yaw), np.cos(desired_yaw - yaw))
        align = np.cos(yaw_error)
        wx, wy = hero["next_wps"]
        d2r = self._lateral_error(x, y, wx, wy)
        e = np.clip(abs(d2r), 0.0, g("lat_clip", 4.0))
        r -= g("k_lat_quadratic", 0.004) * (e * e)
        dist2wp = float(hero["dist2wp"])
        if dist2wp > g("route_dev_start", 8.0):
            r -= g("k_route_dev", 0.006) * (dist2wp - g("route_dev_start", 8.0))
        dprog = self.dist2goal_1 - self.dist2goal
        if dprog > 0 and not (offroad and g("zero_progress_reward_offroad", True)):
            r += g("k_progress", 0.06) * dprog * max(0.0, align)
        if v > 0.3 and not (offroad and g("zero_speed_reward_offroad", True)):
            r += g("k_flow", 0.010) * min(v, g("max_speed_for_flow", 6.0)) * max(0.0, align)
        if e < g("lat_small", 0.8) and abs(yaw_error) < g("yaw_small", 0.12):
            r += g("k_align_bonus", 0.02)
        r += g("k_ttc", 0.03) * self._ttc_shaping(hero["state"], nearby, 30)
        if v < -0.1:
            r += -g("k_reverse", 0.03) * abs(v)
        dyaw = yaw_1 - yaw
        steer_jerk = abs(dyaw - self.last_delta_yaw)
        self.last_delta_yaw = dyaw
        r -= g("k_steer_smooth", 0.003) * abs(dyaw)
        r -= g("k_steer_jerk", 0.01) * steer_jerk
        r += -g("k_smooth", 0.0006) * (abs(v_1 - v) + abs(dyaw))
        r += g("alive_bias", 0.0025)
        return float(np.tanh(r * 1.2))

    # ----------------------------------------------------------------- stats
    def stats_reset(self):
        self.ep_rewards, self.ep_speeds = [], []
        self.ep_comfort = {k: [] for k in COMFORT_KEYS}
        self.ep_viol, self.ep_harsh = [], []
        self.ep_cause = CAUSE_NONE

    def stats_step(self, reward, cause):
        """EpisodeStats.step, stats.py:30-56."""
        self.ep_rewards.append(reward)
        if cause != CAUSE_NONE:
            self.ep_cause = cause
        self.ep_speeds.append(self.ego.v)
        for k in COMFORT_KEYS:
            self.ep_comfort[k].append(abs(float(self.comfort[k])))
        self.ep_viol.append(1.0 if self.comfort_violations() > 0 else 0.0)
        self.ep_harsh.append(1.0 if float(self.comfort["accel_long"]) < -COMFORT_BOUNDS["accel_long"] else 0.0)

    def episode_summary(self):
        """Stats.get_episode_info (per-episode fields), stats.py:127-148."""
        mean = lambda v: float(np.mean(v)) if len(v) else 0.0  # noqa: E731
        out = dict(termination=CAUSE_NAMES[self.ep_cause], length=len(self.ep_rewards),
                   mean_speed=mean(self.ep_speeds), comfort_violation_rate=mean(self.ep_viol),
                   harsh_brake_rate=mean(self.ep_harsh))
        out["return"] = float(np.sum(self.ep_rewards))
        for k in COMFORT_KEYS:
            out[f"mean_abs_{k}"] = mean(self.ep_comfort[k])
        return out

    # ------------------------------------------------------------------ step
    def step(self, gas, steer, brake):
        """CarlaBEV.step minus rendering, carlabev.py:223-231."""
        self.scene_step(gas, steer, brake)
        hit, hit_id, nearby, tile = self.collision_check()
        hero = self.hero_info()
        if self.reward_mode == "carl":
            reward, terminated, cause = self.carl_reward(hit, hit_id, nearby, tile, hero)
        else:
            reward, terminated, cause = self.shaping_reward(hit, hit_id, nearby, tile, hero)
        self.stats_step(reward, cause)
        terminated = cause in TERMINAL_CAUSES  # carlabev.py:177-185
        truncated = cause == CAUSE_MAX_ACTIONS
        self.last = dict(hit=hit, hit_id=hit_id, tile=tile, n_nearby=len(nearby), dist2wp=float(hero["dist2wp"]),
                         cause=cause, nearby=nearby)
        return reward, terminated, truncated, cause

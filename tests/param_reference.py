"""Vectorised float64 restatement of reset / step / observation for ANY ``DDParams`` (TEST-ONLY reference).

``oracle/drone_port.py`` and ``oracle/drone_oracle.c`` hard-code config.py's constants; this module states the same
semantics, in the same statement order as ``drone_port.py`` (thrust through ``_rot``, sequential fuel gating, update,
wrap, then the terminal priority land > ground > fuel > out of bounds > shaping), with every literal replaced by its
``DDParams`` field, for n environments at once as numpy arrays.  The additions the reference lacks are stated as the C
oracle states them: Philox spawns ``min + mulhi32(word, (uint32) count)`` with the words of
``oracle_philox4x32_10`` keyed like ``spawn_draw`` (counter = env id, episode; key = seed), ``max_steps`` truncation,
same-step auto-reset, freeze-after-done, and the episode statistics.

The landing speed test is the reference's ``sqrt(vx^2 + vy^2) > land_speed`` -- not the kernels' pre-rounded squared
threshold -- so that the two can disagree if ``speed2_threshold`` is wrong.

Pinned to the C oracle at the default parameters and to the golden vectors by tests/test_params_cpu.py.
"""
from __future__ import annotations

import numpy as np

from oracle import c_oracle as co

DONE, LANDED, CRASHED, TRUNCATED = 0x01, 0x02, 0x04, 0x08
CAUSE_GROUND, CAUSE_FUEL, CAUSE_OOB = 0x10, 0x20, 0x30
ACT_MAIN, ACT_LEFT, ACT_RIGHT, ACT_SKIP = 0x01, 0x02, 0x04, 0x80
POL_TRACE, POL_RANDOM, POL_BANGBANG = 0, 1, 2


def _rot(x, y, deg):
    # physics.py:16-23
    rad = np.radians(deg)
    c = np.cos(rad)
    s = np.sin(rad)
    return x * c - y * s, x * s + y * c


def _mulhi32(a, b):
    return (np.uint64(a) * np.uint64(b)) >> np.uint64(32)


class RefStats:
    def __init__(self):
        self.episodes = self.landed = self.crashed = self.truncated = self.sum_length = 0
        self.sum_return = 0.0

    def as_tuple(self):
        return (self.episodes, self.landed, self.crashed, self.truncated, self.sum_length)


class ParamRef:
    """n float64 environments under the parameters ``p`` (a ``DDParams``)."""

    def __init__(self, n, p, seed=0, randomize_drone=False, randomize_platform=True, max_steps=0, auto_reset=False,
                 env_id_base=0):
        self.n, self.p = int(n), p
        self.seed, self.env_id_base = int(seed), int(env_id_base)
        self.randomize_drone, self.randomize_platform = bool(randomize_drone), bool(randomize_platform)
        self.max_steps, self.auto_reset = int(max_steps or 0), bool(auto_reset)
        z = lambda: np.zeros(self.n, np.float64)
        self.x, self.y, self.vx, self.vy = z(), z(), z(), z()
        self.angle, self.angvel, self.fuel, self.ret = z(), z(), z(), z()
        self.px, self.py = z(), z()
        self.steps = np.zeros(self.n, np.int32)
        self.episode = np.zeros(self.n, np.uint32)
        self.flags = np.zeros(self.n, np.uint8)
        self.stats = RefStats()

    # ---- reset: game_engine.py:59-93, drone.py:221-238, platform.py:104-114 + Philox spawns ----
    def spawn(self, idx):
        """The spawn coordinates of the next episode of the envs ``idx`` (episode counter not advanced)."""
        p = self.p
        m = len(idx)
        x, y = np.full(m, p.start_x), np.full(m, p.start_y)
        px, py = np.full(m, p.plat_default_x), np.full(m, p.plat_default_y)
        if self.randomize_drone or self.randomize_platform:
            key = (self.seed & 0xffffffff, self.seed >> 32)
            w = np.array([co.philox(((g & 0xffffffff), g >> 32, int(self.episode[i]), 0), key)
                          for i, g in ((i, self.env_id_base + int(i)) for i in idx)], np.uint64).reshape(m, 4)
            if self.randomize_drone:        # np.random.randint(lo, hi + 1)
                x = p.spawn_x_min + _mulhi32(w[:, 0], int(p.spawn_x_count)).astype(np.float64)
                y = p.spawn_y_min + _mulhi32(w[:, 1], int(p.spawn_y_count)).astype(np.float64)
            if self.randomize_platform:     # np.random.randint(lo, hi)
                px = p.plat_x_min + _mulhi32(w[:, 2], int(p.plat_x_count)).astype(np.float64)
                py = p.plat_y_min + _mulhi32(w[:, 3], int(p.plat_y_count)).astype(np.float64)
        return x, y, px, py

    def _reset_idx(self, idx):
        if len(idx) == 0:
            return
        x, y, px, py = self.spawn(idx)
        self.x[idx], self.y[idx], self.px[idx], self.py[idx] = x, y, px, py
        for a in (self.vx, self.vy, self.angle, self.angvel, self.ret):
            a[idx] = 0.0
        self.fuel[idx] = self.p.max_fuel
        self.steps[idx] = 0
        self.flags[idx] = 0
        self.episode[idx] += np.uint32(1)

    def reset(self, mask=None, stride=15):
        idx = np.arange(self.n) if mask is None else np.nonzero(np.asarray(mask))[0]
        self._reset_idx(idx)
        return self.obs(stride)

    def inject(self, x, y, px, py):
        """``g.reset(); g.drone.reset(x, y); g.platform.reset(px, py)`` for every env."""
        self.x[:] = x; self.y[:] = y; self.px[:] = px; self.py[:] = py
        for a in (self.vx, self.vy, self.angle, self.angvel, self.ret):
            a[:] = 0.0
        self.fuel[:] = self.p.max_fuel
        self.steps[:] = 0; self.flags[:] = 0; self.episode += np.uint32(1)

    # ---- observation: game_engine.py:146-177 ----
    def obs(self, stride=15, flags=None):
        p = self.p
        f = self.flags if flags is None else flags
        o = np.zeros((self.n, stride), np.float64)
        dx, dy = self.px - self.x, self.py - self.y
        d = np.sqrt((self.px - self.x) ** 2 + (self.py - self.y) ** 2)
        o[:, 0] = self.x / p.width
        o[:, 1] = self.y / p.height
        o[:, 2] = self.vx / p.vel_norm
        o[:, 3] = self.vy / p.vel_norm
        o[:, 4] = self.angle / p.angle_norm
        o[:, 5] = self.angvel / p.angvel_norm
        o[:, 6] = self.fuel / p.max_fuel
        o[:, 7] = self.px / p.width
        o[:, 8] = self.py / p.height
        o[:, 9] = d / p.width
        o[:, 10] = dx / p.width
        o[:, 11] = dy / p.height
        o[:, 12] = np.sqrt(self.vx ** 2 + self.vy ** 2) / p.vel_norm
        o[:, 13] = (f & LANDED) != 0
        o[:, 14] = (f & CRASHED) != 0
        if stride > 15:
            o[:, 15] = self.steps
        return o

    # ---- step: game_engine.py:95-138 ----
    def _step_live(self, m, act):
        """One DroneGame.step for the envs of boolean mask ``m``; returns (reward, flags) of those envs."""
        p = self.p
        x, y, vx, vy = self.x[m], self.y[m], self.vx[m], self.vy[m]
        angle, angvel, fuel = self.angle[m], self.angvel[m], self.fuel[m]
        px, py = self.px[m], self.py[m]
        a = act[m]
        # drone.py:58-76 -- fuel is re-tested before every thruster
        g = ((a & ACT_MAIN) != 0) & (fuel > 0)
        tx, ty = _rot(0, -p.main_thrust, angle)
        vx = np.where(g, vx + tx, vx); vy = np.where(g, vy + ty, vy); fuel = np.where(g, fuel - p.fuel_main, fuel)
        g = ((a & ACT_LEFT) != 0) & (fuel > 0)
        angvel = np.where(g, angvel - p.side_thrust, angvel); fuel = np.where(g, fuel - p.fuel_side, fuel)
        g = ((a & ACT_RIGHT) != 0) & (fuel > 0)
        angvel = np.where(g, angvel + p.side_thrust, angvel); fuel = np.where(g, fuel - p.fuel_side, fuel)
        fuel = np.maximum(0, fuel)
        # drone.py:88-103 (dt == 1.0)
        vy = vy + p.gravity * 1.0
        vx = vx * p.drag
        vy = vy * p.drag
        x = x + vx * 1.0
        y = y + vy * 1.0
        angle = angle + angvel * 1.0
        angvel = angvel * p.angular_drag
        while (angle > 180).any():                          # physics.py:35-39
            angle = np.where(angle > 180, angle - 360, angle)
        while (angle < -180).any():
            angle = np.where(angle < -180, angle + 360, angle)
        # game_engine.py:185-216 -- priority: land, crash, fuel, oob, shaping
        ox, oy = _rot(0, p.drone_height / 2, angle)        # drone.py:136-137
        bx, by = x + ox, y + oy
        on = (px - p.platform_w / 2 <= bx) & (bx <= px + p.platform_w / 2) & \
             (py - p.platform_h / 2 <= by) & (by <= py + p.platform_h / 2)      # platform.py:57-74
        speed = np.sqrt(vx ** 2 + vy ** 2)                  # drone.py:145
        landing = on & ~(speed > p.land_speed) & (np.abs(angle) <= p.land_angle)
        ground = y > p.height - p.ground_margin              # game_engine.py:254
        fuel_out = fuel <= 0
        mg = p.oob_margin
        oob = (x < -mg) | (x > p.width + mg) | (y < -mg) | (y > p.height + mg)
        d = np.sqrt((px - x) ** 2 + (py - y) ** 2)
        r = p.r_step + (p.shape_offset - d) / p.shape_div
        f = np.zeros(len(x), np.uint8)
        for cond, fl, rt in ((oob, DONE | CRASHED | CAUSE_OOB, p.r_oob), (fuel_out, DONE | CRASHED | CAUSE_FUEL, p.r_fuel),
                             (ground, DONE | CRASHED | CAUSE_GROUND, p.r_crash), (landing, DONE | LANDED, p.r_land)):
            f = np.where(cond, np.uint8(fl), f)
            r = np.where(cond, p.r_step + rt, r)
        self.x[m], self.y[m], self.vx[m], self.vy[m] = x, y, vx, vy
        self.angle[m], self.angvel[m], self.fuel[m] = angle, angvel, fuel
        self.ret[m] += r                                    # game_engine.py:131
        self.steps[m] += 1                                  # game_engine.py:132
        return r, f

    def step(self, actions, stride=15, want_final=False):
        """Batched step with the C oracle's orchestration (oracle_step): returns obs, reward, flags of this step
        (+ the terminal observation of the envs that ended, when ``want_final``)."""
        act = np.asarray(actions, np.uint8)
        reward = np.zeros(self.n)
        out = self.flags.copy()
        m = ((act & ACT_SKIP) == 0) & ((self.flags & DONE) == 0)
        if m.any():
            r, f = self._step_live(m, act)
            trunc = (f == 0) & (self.max_steps > 0) & (self.steps[m] >= self.max_steps)
            f = np.where(trunc, np.uint8(DONE | TRUNCATED), f)
            reward[m] = r
            out[m] = f
            self.flags[m] = f
        fresh = m & ((out & DONE) != 0)
        st = self.stats
        st.episodes += int(fresh.sum())
        st.landed += int((fresh & ((out & LANDED) != 0)).sum())
        st.crashed += int((fresh & ((out & CRASHED) != 0)).sum())
        st.truncated += int((fresh & ((out & TRUNCATED) != 0)).sum())
        st.sum_length += int(self.steps[fresh].sum())
        st.sum_return += float(self.ret[fresh].sum())
        final = None
        if want_final:
            final = np.zeros((self.n, stride))
            final[fresh] = self.obs(stride)[fresh]
        if self.auto_reset:
            self._reset_idx(np.nonzero(fresh)[0])
        obs = self.obs(stride)
        return (obs, reward, out, final) if want_final else (obs, reward, out)

    def rollout(self, T, policy, actions=None, t0=0, stride=15):
        """T steps with the built-in action sources of dd_rollout; returns reward [T,n], done flags [T,n], obs [T,n,stride]
        (the observation AFTER each step)."""
        rew, don, obs = np.zeros((T, self.n)), np.zeros((T, self.n), np.uint8), np.zeros((T, self.n, stride))
        if policy == POL_RANDOM:
            actions = co.random_actions(self.seed, self.env_id_base, t0, T, self.n)
        for t in range(T):
            a = actions[t] if policy != POL_BANGBANG else np.where(self.vy > 1.5, ACT_MAIN, 0).astype(np.uint8)
            obs[t], rew[t], don[t] = self.step(a, stride)
        return rew, don, obs

    # ---- for the float32 comparisons ----
    def threshold_margin(self):
        """Smallest distance of each env's state to a termination threshold, in raw units (px, deg, px/step, fuel)."""
        p = self.p
        ox, oy = _rot(0, p.drone_height / 2, self.angle)
        bx, by = self.x + ox, self.y + oy
        speed = np.sqrt(self.vx ** 2 + self.vy ** 2)
        mg = p.oob_margin
        m = [np.abs(speed - p.land_speed), np.abs(np.abs(self.angle) - p.land_angle),
             np.abs(bx - (self.px - p.platform_w / 2)), np.abs(bx - (self.px + p.platform_w / 2)),
             np.abs(by - (self.py - p.platform_h / 2)), np.abs(by - (self.py + p.platform_h / 2)),
             np.abs(self.y - (p.height - p.ground_margin)), np.abs(self.x + mg), np.abs(self.x - (p.width + mg)),
             np.abs(self.y + mg), np.abs(self.y - (p.height + mg)), np.abs(self.fuel)]
        return np.min(np.stack(m), axis=0)


# ---- the non-default parameter sets the parametrised tests run -------------------------------------------------------
# "hard physics": every field moved.  land_speed 2.7 has an inexact square (speed2_threshold refines it, differently in
# float32 and float64); drone_height 21 and platform_w 101 make the reach halves non-integers; fuel costs are dyadic so
# that the fuel-out step does not depend on the precision, with a small tank so fuel-outs happen.
HARD = dict(
    width=640.0, height=480.0, gravity=0.25, drag=0.985, angular_drag=0.9, drone_height=21.0, main_thrust=0.55,
    side_thrust=0.35, max_fuel=240.0, fuel_main=2.5, fuel_side=0.75, platform_w=101.0, platform_h=15.0,
    land_speed=2.7, land_angle=17.5, oob_margin=40.0, ground_margin=35.0, r_land=80.0, r_crash=-75.0, r_fuel=-40.0,
    r_oob=-30.0, r_step=-0.05, shape_offset=400.0, shape_div=4000.0, start_x=320.0, start_y=80.0,
    plat_default_x=300.0, plat_default_y=390.0, spawn_x_min=60.0, spawn_x_count=521.0, spawn_y_min=30.0,
    spawn_y_count=151.0, plat_x_min=90.0, plat_x_count=461.0, plat_y_min=120.0, plat_y_count=300.0,
    vel_norm=8.0, angle_norm=90.0, angvel_norm=5.0)

# "large world": coordinates around 20,000 px, where one float32 ulp is 1.95e-3 px (the default world stays below 1,024).
LARGE = dict(
    width=40000.0, height=30000.0, start_x=20400.0, start_y=20100.0, plat_default_x=20400.0, plat_default_y=20500.0,
    spawn_x_min=20100.0, spawn_x_count=601.0, spawn_y_min=20050.0, spawn_y_count=201.0,
    plat_x_min=20100.0, plat_x_count=600.0, plat_y_min=20100.0, plat_y_count=450.0)

PARAM_SETS = {"hard": HARD, "large": LARGE}


def make_params(nv, **overrides):
    """config.py's defaults (``nv.default_params()``) with ``overrides`` applied; ``nv`` is the package's _native."""
    p = nv.default_params()
    for k, v in overrides.items():
        if not hasattr(p, k):
            raise KeyError(k)
        setattr(p, k, float(v))
    return p


def world_scale(p):
    """Ratio of the largest coordinate the parameters allow to the default world's (850 px): float32 rounding errors of
    positions, and so the band around a threshold in which float32 and float64 may decide differently, grow with it."""
    return max(1.0, max(p.width + p.oob_margin, p.height + p.oob_margin) / 850.0)

"""gym 0.17-0.19 classic_control envs restated in plain Python, step() as gym writes it (test infrastructure).

They are the independent check of the C envs in oracle/azg_oracle.c, which the engine's envs (csrc/env.cuh) are held to bit for bit:
tests compare the two with the same sine and cosine (sin=det_sin / cos=det_cos are the deterministic ones of the oracle and engine).

* `MountainCarEnv`: classic_control/mountain_car.py.
* `Continuous_MountainCarEnv`: classic_control/continuous_mountain_car.py.
* `AcrobotEnv`: classic_control/acrobot.py with `rk4`, `wrap` and `bound` as gym writes them.  Two departures, both the engine's: the
  square of a float is x * x (gym's x ** 2 calls pow, which is not always correctly rounded), and wrap stops after WRAP_CAP iterations
  per loop (raising oracle.azo.WrapCapReached).
"""
from __future__ import annotations

import math

import numpy as np

from oracle import azo
from oracle.azo import WrapCapReached

WRAP_CAP = 64  # iterations per wrap loop (ACROBOT_WRAP_CAP in csrc/env.cuh and oracle/azg_oracle.c)


class MountainCarEnv:  # gym's class name, which the drop-in search classes recognise
    """gym 0.17-0.19 classic_control/mountain_car.py.  `cos` is math.cos; the engine's bit-exact twin is the deterministic cosine
    (pass cos=det_cos)."""
    min_position, max_position, max_speed = -1.2, 0.6, 0.07
    goal_position, goal_velocity = 0.5, 0
    force, gravity = 0.001, 0.0025

    def __init__(self, state=(-0.5, 0.0), cos=math.cos):
        self.state = np.array(state, dtype=np.float64)
        self.cos = cos

    @property
    def unwrapped(self):
        return self

    def step(self, action):
        position, velocity = self.state
        velocity += (int(action) - 1) * self.force + self.cos(3 * position) * (-self.gravity)
        velocity = np.clip(velocity, -self.max_speed, self.max_speed)
        position += velocity
        position = np.clip(position, self.min_position, self.max_position)
        if position == self.min_position and velocity < 0:
            velocity = 0
        done = bool(position >= self.goal_position and velocity >= self.goal_velocity)
        reward = -1.0
        self.state = (position, velocity)
        return np.array(self.state), reward, done, {}


class Continuous_MountainCarEnv:  # noqa: N801 -- gym's class name, which the drop-in search classes recognise
    """gym 0.17-0.19 classic_control/continuous_mountain_car.py.  The f32 action enters f64 arithmetic exactly (numpy-1.x promotion
    of the reference's pinned numpy; under NEP 50 np.float32 * float would stay f32, hence the explicit float()).  `cos` is math.cos;
    the engine's bit-exact twin is the deterministic cosine (pass cos=det_cos)."""
    min_action, max_action = -1.0, 1.0
    min_position, max_position, max_speed = -1.2, 0.6, 0.07
    goal_position, goal_velocity, power = 0.45, 0, 0.0015

    def __init__(self, state, cos=math.cos):
        self.state = np.array(state, dtype=np.float64)
        self.cos = cos

    @property
    def unwrapped(self):
        return self

    def obs(self):
        return np.array(self.state, dtype=np.float64)

    def step(self, action):
        position, velocity = float(self.state[0]), float(self.state[1])
        a = float(np.asarray(action, dtype=np.float32).ravel()[0])
        force = min(max(a, self.min_action), self.max_action)
        velocity += force * self.power - 0.0025 * self.cos(3 * position)
        if velocity > self.max_speed:
            velocity = self.max_speed
        if velocity < -self.max_speed:
            velocity = -self.max_speed
        position += velocity
        if position > self.max_position:
            position = self.max_position
        if position < self.min_position:
            position = self.min_position
        if position == self.min_position and velocity < 0:
            velocity = 0
        done = bool(position >= self.goal_position and velocity >= self.goal_velocity)
        reward = 0
        if done:
            reward = 100.0
        reward -= math.pow(a, 2) * 0.1
        self.state = np.array([position, velocity], dtype=np.float64)
        return self.obs(), reward, done, {}


def wrap(x, m, M):
    """gym's wrap, with the engine's iteration cap."""
    diff = M - m
    k = 0
    while x > M:
        if k == WRAP_CAP:
            raise WrapCapReached(x)
        x = x - diff
        k += 1
    k = 0
    while x < m:
        if k == WRAP_CAP:
            raise WrapCapReached(x)
        x = x + diff
        k += 1
    return x


def bound(x, m, M=None):
    if M is None:
        M = m[1]
        m = m[0]
    return min(max(x, m), M)


def rk4(derivs, y0, t, *args, **kwargs):
    try:
        Ny = len(y0)
    except TypeError:
        yout = np.zeros((len(t),), np.float64)
    else:
        yout = np.zeros((len(t), Ny), np.float64)
    yout[0] = y0
    for i in np.arange(len(t) - 1):
        thist = t[i]
        dt = t[i + 1] - thist
        dt2 = dt / 2.0
        y0 = yout[i]
        k1 = np.asarray(derivs(y0, thist, *args, **kwargs))
        k2 = np.asarray(derivs(y0 + dt2 * k1, thist + dt2, *args, **kwargs))
        k3 = np.asarray(derivs(y0 + dt2 * k2, thist + dt2, *args, **kwargs))
        k4 = np.asarray(derivs(y0 + dt * k3, thist + dt, *args, **kwargs))
        yout[i + 1] = y0 + dt / 6.0 * (k1 + 2 * k2 + 2 * k3 + k4)
    return yout


class AcrobotEnv:  # gym's class name, which the drop-in search classes recognise
    """gym 0.17-0.19 classic_control/acrobot.py (book dynamics, no torque noise).  `sin` / `cos` default to math's (glibc)."""
    dt = .2
    LINK_LENGTH_1 = 1.
    LINK_LENGTH_2 = 1.
    LINK_MASS_1 = 1.
    LINK_MASS_2 = 1.
    LINK_COM_POS_1 = 0.5
    LINK_COM_POS_2 = 0.5
    LINK_MOI = 1.
    MAX_VEL_1 = 4 * np.pi
    MAX_VEL_2 = 9 * np.pi
    AVAIL_TORQUE = [-1., 0., +1]
    torque_noise_max = 0.
    book_or_nips = "book"

    def __init__(self, state=(0.0, 0.0, 0.0, 0.0), sin=math.sin, cos=math.cos):
        self.state = np.array(state, dtype=np.float64)
        self.sin, self.cos = sin, cos

    @property
    def unwrapped(self):
        return self

    def step(self, a):
        s = self.state
        torque = self.AVAIL_TORQUE[a]
        s_augmented = np.append(s, torque)
        ns = rk4(self._dsdt, s_augmented, [0, self.dt])
        ns = ns[-1]
        ns = ns[:4]
        ns[0] = wrap(ns[0], -np.pi, np.pi)
        ns[1] = wrap(ns[1], -np.pi, np.pi)
        ns[2] = bound(ns[2], -self.MAX_VEL_1, self.MAX_VEL_1)
        ns[3] = bound(ns[3], -self.MAX_VEL_2, self.MAX_VEL_2)
        self.state = ns
        terminal = self._terminal()
        reward = -1. if not terminal else 0.
        return (self._get_ob(), reward, terminal, {})

    def _get_ob(self):
        s = self.state
        return np.array([self.cos(s[0]), self.sin(s[0]), self.cos(s[1]), self.sin(s[1]), s[2], s[3]])

    def _terminal(self):
        s = self.state
        return bool(-self.cos(s[0]) - self.cos(s[1] + s[0]) > 1.)

    def _dsdt(self, s_augmented, t):
        sin, cos, pi = self.sin, self.cos, np.pi
        m1 = self.LINK_MASS_1
        m2 = self.LINK_MASS_2
        l1 = self.LINK_LENGTH_1
        lc1 = self.LINK_COM_POS_1
        lc2 = self.LINK_COM_POS_2
        I1 = self.LINK_MOI
        I2 = self.LINK_MOI
        g = 9.8
        a = s_augmented[-1]
        s = s_augmented[:-1]
        theta1 = s[0]
        theta2 = s[1]
        dtheta1 = s[2]
        dtheta2 = s[3]
        d1 = m1 * lc1 ** 2 + m2 * \
            (l1 ** 2 + lc2 ** 2 + 2 * l1 * lc2 * cos(theta2)) + I1 + I2
        d2 = m2 * (lc2 ** 2 + l1 * lc2 * cos(theta2)) + I2
        phi2 = m2 * lc2 * g * cos(theta1 + theta2 - pi / 2.)
        # gym writes dtheta2 ** 2, dtheta1 ** 2 and d2 ** 2: the engine's convention (DESIGN.md section 6) is the correctly rounded square
        phi1 = - m2 * l1 * lc2 * (dtheta2 * dtheta2) * sin(theta2) \
               - 2 * m2 * l1 * lc2 * dtheta2 * dtheta1 * sin(theta2)  \
            + (m1 * lc1 + m2 * l1) * g * cos(theta1 - pi / 2) + phi2
        # the "book" branch
        ddtheta2 = (a + d2 / d1 * phi1 - m2 * l1 * lc2 * (dtheta1 * dtheta1) * sin(theta2) - phi2) \
            / (m2 * lc2 ** 2 + I2 - (d2 * d2) / d1)
        ddtheta1 = -(d2 * ddtheta2 + phi1) / d1
        return (dtheta1, dtheta2, ddtheta1, ddtheta2, 0.)


def det_cos(x: float) -> float:
    return float(azo.det_eval("cos", np.array([float(x)]), n_threads=1)[0])


def det_sin(x: float) -> float:
    return float(azo.det_eval("sin", np.array([float(x)]), n_threads=1)[0])

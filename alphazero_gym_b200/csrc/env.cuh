// env.cuh -- CartPole-v0 / Pendulum-v0 / MountainCarContinuous-v0 transition functions (gym 0.17.2 / 0.19.0 classic_control,
// third-party to the reference; reached through rl/make_game.py:59-62 and stepped by the search at
// alphazero/search/mcts.py:449 and :686).  Replaces `copy.deepcopy(Env)` + replay from the root
// (mcts.py:443, :680): the hidden state is kept per node and stepped once at expansion.
// All arithmetic is float64 with the rounding sequence of the Python source (built with -fmad=false).
#pragma once
#include "detmath.cuh"

namespace env {

// returns done
__device__ __forceinline__ bool cartpole_step(const double s[4], int action, double o[4], double& reward) {
    const double gravity = 9.8, masscart = 1.0, masspole = 0.1, length = 0.5, force_mag = 10.0, tau = 0.02;
    const double total_mass = masspole + masscart, polemass_length = masspole * length;
    const double theta_thr = 12 * 2 * 3.141592653589793 / 360, x_thr = 2.4;
    double x = s[0], x_dot = s[1], theta = s[2], theta_dot = s[3];
    const double force = action == 1 ? force_mag : -force_mag;
    double sintheta, costheta;
    det::sincos_(theta, sintheta, costheta);
    const double temp = (force + polemass_length * (theta_dot * theta_dot) * sintheta) / total_mass;
    const double thetaacc =
        (gravity * sintheta - costheta * temp) / (length * (4.0 / 3.0 - masspole * (costheta * costheta) / total_mass));
    const double xacc = temp - polemass_length * thetaacc * costheta / total_mass;
    x = x + tau * x_dot;
    x_dot = x_dot + tau * xacc;
    theta = theta + tau * theta_dot;
    theta_dot = theta_dot + tau * thetaacc;
    o[0] = x; o[1] = x_dot; o[2] = theta; o[3] = theta_dot;
    reward = 1.0;
    return x < -x_thr || x > x_thr || theta < -theta_thr || theta > theta_thr;
}

// Python float modulo: result takes the sign of the divisor
__device__ __forceinline__ double py_mod(double a, double b) {
    double r = fmod(a, b);
    if (r != 0.0) {
        if ((b < 0) != (r < 0)) r += b;
    } else {
        r = copysign(0.0, b);
    }
    return r;
}

// returns done (always false); reward is the raw env reward (-costs)
__device__ __forceinline__ bool pendulum_step(double th, double thdot, float action, double& newth, double& newthdot,
                                              double& reward) {
    const double max_speed = 8, dt = 0.05, g = 10.0, m = 1.0, l = 1.0, pi = 3.141592653589793;
    const float uf = action < -2.0f ? -2.0f : (action > 2.0f ? 2.0f : action);  // np.clip on the f32 action
    const double u = (double)uf;  // numpy-1.x promotion of the f32 torque (SURVEY 8c)
    const double an = py_mod(th + pi, 2 * pi) - pi;
    const double costs = an * an + 0.1 * (thdot * thdot) + 0.001 * (u * u);
    double nd = thdot + (-3 * g / (2 * l) * det::sin_(th + pi) + 3.0 / (m * (l * l)) * u) * dt;
    newth = th + nd * dt;
    nd = nd < -max_speed ? -max_speed : (nd > max_speed ? max_speed : nd);
    newthdot = nd;
    reward = -costs;
    return false;
}

__device__ __forceinline__ float4 pendulum_obs(double th, double thdot) {
    double s, c;
    det::sincos_(th, s, c);
    return make_float4((float)c, (float)s, (float)thdot, 0.0f);
}

// MountainCarContinuous-v0 (gym 0.17-0.19 classic_control/continuous_mountain_car.py); returns done.  The f32 action enters f64
// arithmetic exactly (numpy-1.x promotion, as for Pendulum); the clips are Python's max / min (a NaN passes, -0 stays -0); the
// reward uses the unclipped action, and 0 - x with the int 0 is 0.0 - x (+0 for a zero action).
__device__ __forceinline__ bool mountain_car_step(double pos, double vel, float action, double& newpos, double& newvel, double& reward) {
    const double min_position = -1.2, max_position = 0.6, max_speed = 0.07, goal_position = 0.45, power = 0.0015;
    const double a = (double)action;
    double force = -1.0 > a ? -1.0 : a;  // min(max(action[0], min_action), max_action)
    force = 1.0 < force ? 1.0 : force;
    vel = vel + (force * power - 0.0025 * det::cos_(3 * pos));
    if (vel > max_speed) vel = max_speed;
    if (vel < -max_speed) vel = -max_speed;
    pos = pos + vel;
    if (pos > max_position) pos = max_position;
    if (pos < min_position) pos = min_position;
    if (pos == min_position && vel < 0) vel = 0.0;
    const bool done = pos >= goal_position && vel >= 0.0;
    reward = (done ? 100.0 : 0.0) - (a * a) * 0.1;  // math.pow(action[0], 2) of an f32 is exact in f64
    newpos = pos;
    newvel = vel;
    return done;
}

// MountainCar-v0 (gym 0.17-0.19 classic_control/mountain_car.py); returns done.  The right-hand side of `velocity +=` is summed
// first; (action - 1) * force is an int times a float (-0.001, +0.0 or 0.001); np.clip passes a NaN and keeps -0; the left wall stores
// the int 0 (+0 from then on); done is false for a NaN state; the reward is -1.0 on every step, the terminating one included.
__device__ __forceinline__ bool mountain_car_step(double pos, double vel, int action, double& newpos, double& newvel, double& reward) {
    const double min_position = -1.2, max_position = 0.6, max_speed = 0.07, goal_position = 0.5, force = 0.001, gravity = 0.0025;
    vel = vel + ((double)(action - 1) * force + det::cos_(3 * pos) * -gravity);
    vel = vel < -max_speed ? -max_speed : (vel > max_speed ? max_speed : vel);
    pos = pos + vel;
    pos = pos < min_position ? min_position : (pos > max_position ? max_position : pos);
    if (pos == min_position && vel < 0) vel = 0.0;
    newpos = pos;
    newvel = vel;
    reward = -1.0;
    return pos >= goal_position && vel >= 0.0;
}

// Acrobot-v1 (gym 0.17-0.19 classic_control/acrobot.py, book dynamics, no torque noise).  Every operation is f64 in the source's
// left-to-right order; x ** 2 of a float is x * x; sin / cos are the deterministic ones, one sincos_ per distinct argument.
//
// wrap(x, -pi, pi) is gym's pair of unbounded while loops.  Each loop here stops after ACROBOT_WRAP_CAP iterations and sets `capped`
// (the search then fails with ERR_WRAP) instead of spinning on an infinite or huge angle.  Stepped from inside gym's box (angles in
// [-pi, pi], |dtheta1| <= 4 pi, |dtheta2| <= 9 pi) an angle needs at most 5 turns (DESIGN.md section 6), so the cap never changes
// a result gym can produce.  A NaN passes through wrap and bound as it does in gym.
#define ACROBOT_WRAP_CAP 64
__device__ __forceinline__ void acrobot_dsdt(const double s[4], double a, double d[4]) {
    const double m1 = 1.0, m2 = 1.0, l1 = 1.0, lc1 = 0.5, lc2 = 0.5, I1 = 1.0, I2 = 1.0, g = 9.8, pi = 3.141592653589793;
    const double theta1 = s[0], theta2 = s[1], dtheta1 = s[2], dtheta2 = s[3];
    double s2, c2;
    det::sincos_(theta2, s2, c2);
    const double d1 = m1 * (lc1 * lc1) + m2 * (l1 * l1 + lc2 * lc2 + 2 * l1 * lc2 * c2) + I1 + I2;
    const double d2 = m2 * (lc2 * lc2 + l1 * lc2 * c2) + I2;
    const double phi2 = m2 * lc2 * g * det::cos_(theta1 + theta2 - pi / 2.);
    const double phi1 = -m2 * l1 * lc2 * (dtheta2 * dtheta2) * s2 - 2 * m2 * l1 * lc2 * dtheta2 * dtheta1 * s2 +
                        (m1 * lc1 + m2 * l1) * g * det::cos_(theta1 - pi / 2) + phi2;
    const double ddtheta2 = (a + d2 / d1 * phi1 - m2 * l1 * lc2 * (dtheta1 * dtheta1) * s2 - phi2) / (m2 * (lc2 * lc2) + I2 - (d2 * d2) / d1);
    const double ddtheta1 = -(d2 * ddtheta2 + phi1) / d1;
    d[0] = dtheta1; d[1] = dtheta2; d[2] = ddtheta1; d[3] = ddtheta2;
}
__device__ __forceinline__ double acrobot_wrap(double x, bool& capped) {
    const double pi = 3.141592653589793, diff = pi - -pi;
    for (int k = 0; x > pi; ++k) {
        if (k == ACROBOT_WRAP_CAP) { capped = true; return x; }
        x = x - diff;
    }
    for (int k = 0; x < -pi; ++k) {
        if (k == ACROBOT_WRAP_CAP) { capped = true; return x; }
        x = x + diff;
    }
    return x;
}
// bound(x, m, M) = min(max(x, m), M) with Python's builtins: a NaN passes, -0 stays -0
__device__ __forceinline__ double acrobot_bound(double x, double m, double M) {
    x = m > x ? m : x;
    return M < x ? M : x;
}
// returns terminal; reward -1.0 before the goal, 0.0 at it.  The torque (the fifth RK4 component) has derivative 0, so it stays exact.
__device__ __forceinline__ bool acrobot_step(const double s[4], int action, double o[4], double& reward, bool& capped) {
    const double dt = .2, pi = 3.141592653589793, MAX_VEL_1 = 4 * pi, MAX_VEL_2 = 9 * pi;
    const double torque = action == 0 ? -1.0 : (action == 1 ? 0.0 : 1.0);
    const double dt2 = dt / 2.0;
    double k1[4], k2[4], k3[4], k4[4], y[4];
    acrobot_dsdt(s, torque, k1);
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = s[i] + dt2 * k1[i];
    acrobot_dsdt(y, torque, k2);
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = s[i] + dt2 * k2[i];
    acrobot_dsdt(y, torque, k3);
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = s[i] + dt * k3[i];
    acrobot_dsdt(y, torque, k4);
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = s[i] + dt / 6.0 * (k1[i] + 2 * k2[i] + 2 * k3[i] + k4[i]);
    o[0] = acrobot_wrap(o[0], capped);
    o[1] = acrobot_wrap(o[1], capped);
    o[2] = acrobot_bound(o[2], -MAX_VEL_1, MAX_VEL_1);
    o[3] = acrobot_bound(o[3], -MAX_VEL_2, MAX_VEL_2);
    const bool terminal = -det::cos_(o[0]) - det::cos_(o[1] + o[0]) > 1.;
    reward = terminal ? 0.0 : -1.0;
    return terminal;
}
// _get_ob: cos / sin of both angles and both velocities, computed in f64 and rounded to f32 per entry
__device__ __forceinline__ void acrobot_obs(const double s[4], float x[6]) {
    double s0, c0, s1, c1;
    det::sincos_(s[0], s0, c0);
    det::sincos_(s[1], s1, c1);
    x[0] = (float)c0; x[1] = (float)s0; x[2] = (float)c1; x[3] = (float)s1; x[4] = (float)s[2]; x[5] = (float)s[3];
}

// The env of a search as a compile-time type.  S is the network input width, HS the width of the hidden state the tree keeps per node
// (HS doubles; the discrete state table has room for 4).  Continuous: the hidden state is two doubles (CRow sector 1), the network input
// the first S lanes of a float4.  Discrete: A actions, the row layout follows (DRow for 2, D3Row for 3).  CartPole names the discrete
// tree in the kernels that serve both variants.
//
// The three-action envs also give the tree's view of the env on hidden-state arrays: expand (one env step; `capped`: a wrap loop reached
// its cap) and input (the network input as XW = ceil(S / 4) float4, unused lanes 0); Acrobot's reset takes four uniforms.
struct CartPole {
    static constexpr int S = 4, HS = 4, A = 2;
    static constexpr bool DISCRETE = true;
};
struct MountainCar {
    static constexpr int S = 2, HS = 2, A = 3, XW = 1;
    static constexpr bool DISCRETE = true;
    static __device__ __forceinline__ bool step(double pos, double vel, int a, double& npos, double& nvel, double& r) {
        return mountain_car_step(pos, vel, a, npos, nvel, r);
    }
    static __device__ __forceinline__ float4 obs(double pos, double vel) { return make_float4((float)pos, (float)vel, 0.0f, 0.0f); }
    // Env.reset: position ~ U(-0.6, -0.4), velocity +0 (the same formula as MountainCarContinuous)
    static __device__ __forceinline__ void reset(double u0, double, double& pos, double& vel) {
        pos = -0.6 + (-0.4 - -0.6) * u0;
        vel = 0.0;
    }
    static __device__ __forceinline__ bool expand(const double* s, int a, double* o, double& r, bool&) {
        return step(s[0], s[1], a, o[0], o[1], r);
    }
    static __device__ __forceinline__ void input(const double* s, float4* x) { x[0] = obs(s[0], s[1]); }
};
struct Acrobot {
    static constexpr int S = 6, HS = 4, A = 3, XW = 2;
    static constexpr bool DISCRETE = true;
    static __device__ __forceinline__ bool expand(const double* s, int a, double* o, double& r, bool& capped) {
        return acrobot_step(s, a, o, r, capped);
    }
    static __device__ __forceinline__ void input(const double* s, float4* x) {
        float v[6];
        acrobot_obs(s, v);
        x[0] = make_float4(v[0], v[1], v[2], v[3]);
        x[1] = make_float4(v[4], v[5], 0.0f, 0.0f);
    }
    // Env.reset: the state ~ U(-0.1, 0.1)^4
    static __device__ __forceinline__ void reset(const double* u, double* s) {
        for (int k = 0; k < 4; ++k) s[k] = -0.1 + (0.1 - -0.1) * u[k];
    }
};
struct Pendulum {
    static constexpr int S = 3, HS = 2;
    static constexpr bool DISCRETE = false;
    static __device__ __forceinline__ bool step(double th, double thdot, float a, double& nth, double& nthdot, double& r) {
        return pendulum_step(th, thdot, a, nth, nthdot, r);
    }
    static __device__ __forceinline__ float4 obs(double th, double thdot) { return pendulum_obs(th, thdot); }
    // Env.reset from the uniforms u0, u1: th ~ U(-pi, pi), thdot ~ U(-1, 1)
    static __device__ __forceinline__ void reset(double u0, double u1, double& th, double& thdot) {
        const double pi = 3.141592653589793;
        th = -pi + (pi - -pi) * u0;
        thdot = -1.0 + (1.0 - -1.0) * u1;
    }
};
struct MountainCarContinuous {
    static constexpr int S = 2, HS = 2;
    static constexpr bool DISCRETE = false;
    static __device__ __forceinline__ bool step(double pos, double vel, float a, double& npos, double& nvel, double& r) {
        return mountain_car_step(pos, vel, a, npos, nvel, r);
    }
    static __device__ __forceinline__ float4 obs(double pos, double vel) { return make_float4((float)pos, (float)vel, 0.0f, 0.0f); }
    // Env.reset: position ~ U(-0.6, -0.4), velocity +0
    static __device__ __forceinline__ void reset(double u0, double, double& pos, double& vel) {
        pos = -0.6 + (-0.4 - -0.6) * u0;
        vel = 0.0;
    }
};

// actions of a discrete env, 0 for a continuous one
template <class ENV>
__host__ __device__ constexpr int actions_of() {
    if constexpr (ENV::DISCRETE) return ENV::A;
    else return 0;
}
// whether an env's search writes three-action rows (D3Row)
template <class ENV>
__host__ __device__ constexpr bool row3() { return actions_of<ENV>() == 3; }

}  // namespace env

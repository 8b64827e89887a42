// selfplay.cuh -- the environment side of one self-play step, batched: final action from the root statistics, the real
// env step, episode bookkeeping and reset, discrete tree reuse.  One thread per environment.
//
// Reference (per environment, per step): run_continuous.py:117-142 / run_discrete.py:100-122 --
//   action, s, actions, counts, Qs, V = agent.act(Env)         agents.py:492-537 (actions[counts.argmax()]),
//                                                              agents.py:257-303 (stable_normalizer + np.random.choice / argmax)
//   buffer.store((s, actions, counts, Qs, V))                  buffers.py:61
//   state, reward, terminal, _ = Env.step(action)
//   terminal or t == max_episode_length - 1  ->  Env.reset(), agent.reset_mcts(state)
//   else continuous: agent.reset_mcts(state) (no tree reuse)   run_continuous.py:142
//        discrete:   agent.mcts_forward(action, state)         run_discrete.py:122 -> mcts.py:495-526; evaluation(root) re-creates
//                                                              the root's edges, so only root.n survives (SURVEY 7-7)
// Randomness: the engine is re-keyed for every step (azg_selfplay_step); stream 2 = the discrete agent's action draw,
// stream 3 = Env.reset (gym: CartPole U(-0.05, 0.05)^4, Pendulum th ~ U(-pi, pi), thdot ~ U(-1, 1), MountainCarContinuous and
// MountainCar position ~ U(-0.6, -0.4), velocity 0, Acrobot U(-0.1, 0.1)^4).
#pragma once
#include "common.cuh"
#include "env.cuh"

struct SelfPlayParams {
    int32_t B, cmax, max_episode_length, deterministic, by_value;
    double temperature;
    int64_t tree_id0;
    const uint64_t* seedp;
    // state (in/out)
    double* env_state;   // [B][HS]  (CartPole and Acrobot 4; MountainCar and the continuous envs 2)
    int32_t* ep_step;    // [B]
    int32_t* episode;    // [B]
    int32_t* root_n;     // [B] discrete
    // root results of this step's search (in) = the replay row
    const float* actions;
    const int32_t* counts;
    const double* Q;
    const int32_t* n_children;
    // outputs
    float* obs;          // [B][S] observation the search started from (S = 6 | 4 | 3 | 2)
    float* action_taken; // [B]
    double* reward;      // [B]
    int32_t* done;       // [B]
    // discrete tree tables (root.n carry-over)
    const DRow* drows;
    int32_t R;
    int32_t* err;        // ERR_WRAP (Acrobot's real env step)
};

__device__ __forceinline__ double u32_to_unit_f64(uint32_t x) { return ((double)x + 0.5) * 2.3283064365386963e-10; }

template <class ENV>
__global__ void k_selfplay_continuous(const SelfPlayParams p) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p.B) return;
    const int nk = p.n_children[t];
    const float* act = p.actions + (size_t)t * p.cmax;
    int best = 0;
    if (p.by_value) {  // final_selection == "max_value": Q.argmax()
        const double* q = p.Q + (size_t)t * p.cmax;
        for (int j = 1; j < nk; ++j) best = q[j] > q[best] ? j : best;
    } else {           // counts.argmax(): first maximum (agents.py:533)
        const int32_t* c = p.counts + (size_t)t * p.cmax;
        for (int j = 1; j < nk; ++j) best = c[j] > c[best] ? j : best;
    }
    const float a = act[best];
    const double th = p.env_state[(size_t)t * 2], thdot = p.env_state[(size_t)t * 2 + 1];
    const float4 ob = ENV::obs(th, thdot);
    p.obs[(size_t)t * ENV::S] = ob.x; p.obs[(size_t)t * ENV::S + 1] = ob.y;
    if (ENV::S > 2) p.obs[(size_t)t * ENV::S + 2] = ob.z;
    double nth, nthdot, rew;
    const bool term = ENV::step(th, thdot, a, nth, nthdot, rew);
    const int step = p.ep_step[t] + 1;
    const bool done = term || step >= p.max_episode_length;
    if (done) {  // Env.reset()
        const int ep = p.episode[t] + 1;
        const u32x4 r = rng_block(__ldg(p.seedp), p.tree_id0 + t, 3, ep, 0);
        ENV::reset(u32_to_unit_f64(r.x), u32_to_unit_f64(r.y), nth, nthdot);
        p.episode[t] = ep;
    }
    p.ep_step[t] = done ? 0 : step;
    p.env_state[(size_t)t * 2] = nth;
    p.env_state[(size_t)t * 2 + 1] = nthdot;
    p.action_taken[t] = a;
    p.reward[t] = rew;
    p.done[t] = done ? 1 : 0;
}

template <class ENV>
__global__ void k_selfplay_discrete(const SelfPlayParams p) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p.B) return;
    constexpr int A = ENV::A;
    if constexpr (A == 2) {
        // stable_normalizer (helpers.py:9-27): x = (x / max(x)) ** temp; pi = |x / sum(x)|
        double x[2];
        if (p.by_value) { x[0] = p.Q[(size_t)t * p.cmax]; x[1] = p.Q[(size_t)t * p.cmax + 1]; }
        else { x[0] = (double)p.counts[(size_t)t * p.cmax]; x[1] = (double)p.counts[(size_t)t * p.cmax + 1]; }
        const double mx = x[0] > x[1] ? x[0] : x[1];
        for (int i = 0; i < A; ++i) {
            x[i] = x[i] / mx;
            if (p.temperature != 1.0) x[i] = pow(x[i], p.temperature);  // helpers.py:26; pi itself is bit-pinned for temperature == 1 only
        }
        const double sum = x[0] + x[1];
        const double pi0 = fabs(x[0] / sum), pi1 = fabs(x[1] / sum);
        int a;
        if (p.deterministic) {
            a = pi1 > pi0 ? 1 : 0;  // pi.argmax()
        } else {  // np.random.choice(len(pi), p=pi): cdf = cumsum(p) / cdf[-1]; searchsorted(cdf, u, side="right")
            const double u = u32_to_unit_f64(rng_block(__ldg(p.seedp), p.tree_id0 + t, 2, 0, 0).x);
            const double c1 = pi0 + pi1;
            const double cdf0 = pi0 / c1;
            a = u < cdf0 ? 0 : 1;
        }
        double s[4], o[4], rew;
        for (int k = 0; k < 4; ++k) {
            s[k] = p.env_state[(size_t)t * 4 + k];
            p.obs[(size_t)t * 4 + k] = (float)s[k];
        }
        const bool term = env::cartpole_step(s, a, o, rew);
        const int step = p.ep_step[t] + 1;
        const bool done = term || step >= p.max_episode_length;
        int root_n = 0;
        if (done) {  // Env.reset() + reset_mcts
            const int ep = p.episode[t] + 1;
            const u32x4 r = rng_block(__ldg(p.seedp), p.tree_id0 + t, 3, ep, 0);
            o[0] = -0.05 + (0.05 - -0.05) * u32_to_unit_f64(r.x);
            o[1] = -0.05 + (0.05 - -0.05) * u32_to_unit_f64(r.y);
            o[2] = -0.05 + (0.05 - -0.05) * u32_to_unit_f64(r.z);
            o[3] = -0.05 + (0.05 - -0.05) * u32_to_unit_f64(r.w);
            p.episode[t] = ep;
        } else {  // mcts_forward: the chosen child becomes the root and keeps its visit count (mcts.py:510-524)
            const DRow* rows = p.drows + (size_t)t * p.R;
            const uint16_t child = rows[0].child[a];
            root_n = child == DROW_NONE ? 0 : rows[child].node_n;
        }
        p.ep_step[t] = done ? 0 : step;
        p.root_n[t] = root_n;
        for (int k = 0; k < 4; ++k) p.env_state[(size_t)t * 4 + k] = o[k];
        p.action_taken[t] = (float)a;
        p.reward[t] = rew;
        p.done[t] = done ? 1 : 0;
    } else {
        // stable_normalizer over the A counts (or Qs); np.max, then np.sum (sequential for n < 8)
        double x[A];
        for (int i = 0; i < A; ++i) x[i] = p.by_value ? p.Q[(size_t)t * p.cmax + i] : (double)p.counts[(size_t)t * p.cmax + i];
        double mx = x[0];
        for (int i = 1; i < A; ++i) mx = x[i] > mx ? x[i] : mx;
        double sum = 0.0;
        for (int i = 0; i < A; ++i) {
            x[i] = x[i] / mx;
            if (p.temperature != 1.0) x[i] = pow(x[i], p.temperature);
            sum += x[i];
        }
        double pi[A];
        for (int i = 0; i < A; ++i) pi[i] = fabs(x[i] / sum);
        int a = 0;
        if (p.deterministic) {
            for (int i = 1; i < A; ++i) a = pi[i] > pi[a] ? i : a;  // pi.argmax(): the first maximum
        } else {  // np.random.choice: cdf = cumsum(pi); cdf /= cdf[-1]; searchsorted(cdf, u, side="right")
            const double u = u32_to_unit_f64(rng_block(__ldg(p.seedp), p.tree_id0 + t, 2, 0, 0).x);
            double cdf[A];
            cdf[0] = pi[0];
            for (int i = 1; i < A; ++i) cdf[i] = cdf[i - 1] + pi[i];
            const double last = cdf[A - 1];
            for (int i = 0; i < A - 1; ++i) a += (u >= cdf[i] / last) ? 1 : 0;
        }
        // the env step, Env.reset() + reset_mcts when done, else mcts_forward: the chosen child keeps its visit count.  MountainCar's
        // two-wide state stays in scalars as it always was (which keeps that kernel's code unchanged); wider hidden states in arrays.
        double rew;
        bool done;
        int root_n = 0;
        if constexpr (ENV::HS == 2) {
            const double pos = p.env_state[(size_t)t * 2], vel = p.env_state[(size_t)t * 2 + 1];
            const float4 ob = ENV::obs(pos, vel);
            p.obs[(size_t)t * 2] = ob.x; p.obs[(size_t)t * 2 + 1] = ob.y;
            double npos, nvel;
            const bool term = ENV::step(pos, vel, a, npos, nvel, rew);
            const int step = p.ep_step[t] + 1;
            done = term || step >= p.max_episode_length;
            if (done) {
                const int ep = p.episode[t] + 1;
                const u32x4 r = rng_block(__ldg(p.seedp), p.tree_id0 + t, 3, ep, 0);
                ENV::reset(u32_to_unit_f64(r.x), u32_to_unit_f64(r.y), npos, nvel);
                p.episode[t] = ep;
            } else {
                const D3Row* rows = reinterpret_cast<const D3Row*>(p.drows) + (size_t)t * p.R;
                const uint16_t child = rows[0].child[a];
                root_n = child == DROW_NONE ? 0 : rows[child].node_n;
            }
            p.ep_step[t] = done ? 0 : step;
            p.root_n[t] = root_n;
            p.env_state[(size_t)t * 2] = npos;
            p.env_state[(size_t)t * 2 + 1] = nvel;
        } else {
            constexpr int HS = ENV::HS, S = ENV::S;
            double h[HS], o[HS];
#pragma unroll
            for (int k = 0; k < HS; ++k) h[k] = p.env_state[(size_t)t * HS + k];
            float4 ob[ENV::XW];
            ENV::input(h, ob);
#pragma unroll
            for (int k = 0; k < S; ++k) p.obs[(size_t)t * S + k] = reinterpret_cast<const float*>(ob)[k];
            bool capped = false;
            const bool term = ENV::expand(h, a, o, rew, capped);
            if (capped) atomicOr(p.err, ERR_WRAP);
            const int step = p.ep_step[t] + 1;
            done = term || step >= p.max_episode_length;
            if (done) {
                const int ep = p.episode[t] + 1;
                const u32x4 r = rng_block(__ldg(p.seedp), p.tree_id0 + t, 3, ep, 0);
                const double u[4] = {u32_to_unit_f64(r.x), u32_to_unit_f64(r.y), u32_to_unit_f64(r.z), u32_to_unit_f64(r.w)};
                ENV::reset(u, o);
                p.episode[t] = ep;
            } else {
                const D3Row* rows = reinterpret_cast<const D3Row*>(p.drows) + (size_t)t * p.R;
                const uint16_t child = rows[0].child[a];
                root_n = child == DROW_NONE ? 0 : rows[child].node_n;
            }
            p.ep_step[t] = done ? 0 : step;
            p.root_n[t] = root_n;
#pragma unroll
            for (int k = 0; k < HS; ++k) p.env_state[(size_t)t * HS + k] = o[k];
        }
        p.action_taken[t] = (float)a;
        p.reward[t] = rew;
        p.done[t] = done ? 1 : 0;
    }
}

__global__ void k_set_seed(uint64_t* d, uint64_t v) { *d = v; }

/*
 * azg.h -- C ABI of the B200-native batched MCTS engine (libazg.so).
 *
 * This is the drop-in boundary for the search hot path of timoklein/alphazero-gym.  The reference has
 * no FFI: its seam is the Python class chosen by Hydra `_target_` (config/mcts/MCTSDiscrete.yaml:2,
 * config/mcts/MCTSContinuous.yaml:2) and built by the agent (alphazero/agent/agents.py:82).  The host
 * side (alphazero_gym_b200/search/mcts.py) keeps that class interface and calls these entry points
 * through ctypes with raw pointers -- no torch types cross this boundary.  INTEGRATION.md shows the
 * binding a reference maintainer would add.
 *
 * Conventions: every function returns 0 on success and a negative AZG_E* code on failure, with a
 * message available from azg_last_error() (thread-local).  No exceptions cross the boundary.  One engine
 * per GPU; calls on one handle are stream-ordered and not thread-safe.  `stream` is a cudaStream_t
 * passed as void* (NULL = the legacy default stream).  Pointers named d_* are device pointers owned by
 * the caller, h_* are host pointers.  There is no CPU fallback: without a CUDA device azg_create fails.
 */
#ifndef AZG_H
#define AZG_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AZG_OK 0
#define AZG_EINVAL -1      /* bad argument / unsupported configuration */
#define AZG_ECUDA -2       /* CUDA runtime error (message has the cudaError string) */
#define AZG_ETERMINAL -3   /* "Can't do tree search from a terminal node" (mcts.py:382-383, :599-600) */
#define AZG_ENAN -4        /* NaN met in a UCT vector (helpers.py:47-48 only warns; we refuse) */
#define AZG_ECAPACITY -5   /* tree arena / child fan-out capacity exceeded */
#define AZG_EWRAP -6       /* Acrobot-v1: an angle needed more than 64 iterations of gym's wrap loop (an infinite or huge angle, on
                              which gym would loop for that long or forever); the search's results are not gym's */

#define AZG_DISCRETE 0   /* MCTSDiscrete  + CartPole-v0 dynamics (or, with AZG_FLAG_ENV_MOUNTAIN_CAR, MountainCar-v0; with AZG_FLAG_ENV_ACROBOT,
                            Acrobot-v1) + DiscretePolicy */
#define AZG_CONTINUOUS 1 /* MCTSContinuous + Pendulum-v0 (or, with AZG_FLAG_ENV_MOUNTAIN_CAR_CONTINUOUS, MountainCarContinuous-v0)
                           dynamics + DiagonalNormal/GMM policy */

#define AZG_ACT_RELU 0
#define AZG_ACT_ELU 1
/* the other entries of the reference's activation map (alphazero/network/utils.py:5-14); FP32 evaluation kernel only */
#define AZG_ACT_LEAKYRELU 2 /* nn.LeakyReLU(): x > 0 ? x : 0.01 x */
#define AZG_ACT_RELU6 3     /* nn.ReLU6() */
#define AZG_ACT_SILU 4      /* nn.SiLU(), config names "swish" and "silu" */
#define AZG_ACT_HARDSWISH 5 /* nn.Hardswish() */

#define AZG_VT_OFF_POLICY 0 /* mcts.py:131 */
#define AZG_VT_ON_POLICY 1  /* mcts.py:111 */
#define AZG_VT_GREEDY 2     /* mcts.py:133-173 */

/* Constructor arguments of the reference classes (mcts.py:316-327 MCTSDiscrete, :537-549
 * MCTSContinuous) plus what `model` implies (policies.py:806 make_policy) and engine capacity. */
typedef struct azg_config {
    int32_t variant;        /* AZG_DISCRETE | AZG_CONTINUOUS */
    int32_t max_rollouts;   /* capacity: largest n_rollouts a search call may ask for */
    int32_t max_trees;      /* capacity: largest batch B */
    int32_t num_actions;    /* discrete: 2 (CartPole), 3 (MountainCar-v0, Acrobot-v1) */
    int32_t num_components; /* continuous: K mixture components (1 = DiagonalNormalPolicy) */
    int32_t state_dim;      /* network input width: 4 CartPole, 3 Pendulum, 2 MountainCarContinuous and MountainCar, 6 Acrobot */
    int32_t hidden;         /* hidden width (all hidden layers equal; 128 in both shipped configs) */
    int32_t n_hidden;       /* hidden layers: 2 (DiscretePolicy.yaml) / 3 (ContinuousPolicy.yaml) */
    int32_t activation;     /* AZG_ACT_* */
    int32_t v_target;       /* AZG_VT_* (V_target_policy) */
    int32_t puct_f32;       /* 1: prior*c_uct rounded to f32 as numpy>=2 does (mcts.py:484); 0: f64 */
    int32_t device;         /* CUDA device ordinal */
    double c_uct, gamma, epsilon, c_pw, kappa;
    float action_bound, log_std_min, log_std_max;
    uint32_t flags;         /* AZG_FLAG_* */
    uint64_t seed;          /* Philox key for tie-break / eps-greedy / action-noise streams */
} azg_config;

#define AZG_FLAG_NO_GRAPH 1u /* launch kernels directly instead of replaying a captured CUDA graph */
#define AZG_FLAG_EVAL_Q8 2u  /* evaluate the hidden x hidden layers on the tensor cores (tcgen05.mma kind::i8) as exact
                                int8-sliced fixed-point products instead of FP32 FMA; needs hidden = 128, n_hidden in {2,3}.
                                Deterministic and bit-reproducible by the CPU oracle (AZO_EVAL_Q8); V error vs an f64
                                evaluation is ~2x that of the FP32 path, well inside the 1e-5 parity tolerance. */

#define AZG_FLAG_FUSED 4u    /* with AZG_FLAG_EVAL_Q8, both variants (CartPole and Pendulum): run the whole search (root evaluation, every
                                simulation's backup + select + expansion + leaf evaluation) in ONE persistent kernel per chunk of
                                trees; a CTA owns its trees for the whole search.  Three kernels, chosen by batch size and variant
                                (engine.cu launch_fused_t; azg_fused_stats out[5] says which ran): four independent warpgroups per SM,
                                each thread owning its tree's step and its row of the evaluation (>= 3 full tiles per SM); a CTA
                                alternating an evaluation phase and a tree phase (thinner batches); and, for the discrete tree, the
                                same with the CTA's trees RESIDENT IN SHARED MEMORY for the whole search when they fit (BASELINE
                                config 3: 28 CartPole trees per SM).  Same arithmetic, same results bit for bit as the
                                per-simulation launches. */

#define AZG_FLAG_RNG_MT19937 8u /* un-shimmed compatibility: every random number comes from the generators the reference itself uses,
                                   seeded per tree at the start of every search like random.seed(seed + global tree id) and
                                   torch.manual_seed(seed + global tree id).  Tie-break / eps-greedy draws: CPython's MT19937
                                   (init_by_array seeding; random(), choice and randint with CPython's algorithms; helpers.py:50-51,
                                   mcts.py:190-192).  Continuous variant additionally: the action noise of model.sample_action
                                   (policies.py:656-669, :488-499) from torch's CPU generator -- mt19937 + 53-bit uniforms, the
                                   exponential race of torch.multinomial(probs, 1), Box-Muller pairs with the cached sine of
                                   torch.normal -- so that a reference run with its stock `random` module and un-wrapped torch is
                                   reproduced (goldens tests/golden/cartpole_mt_*, pendulum_mt_*).  The continuous variant runs
                                   this mode with one launch per simulation (no AZG_FLAG_FUSED). */

#define AZG_FLAG_ENV_MOUNTAIN_CAR_CONTINUOUS 16u /* continuous variant only, with state_dim 2: the search steps MountainCarContinuous-v0
                                   (gym 0.17-0.19 continuous_mountain_car.py) instead of Pendulum-v0.  Hidden state (position,
                                   velocity), network input (float)position, (float)velocity; an episode ends at the goal, so
                                   expanded nodes can be terminal (V = 0).  The search reward is r / 16.2736044 as for every
                                   continuous search (mcts.py:687).  Every schedule, every other flag and the row, control-block and
                                   result layouts are those of the Pendulum search. */
#define AZG_FLAG_ENV_MOUNTAIN_CAR 32u /* discrete variant only, with num_actions 3 and state_dim 2 (not with
                                   AZG_FLAG_ENV_MOUNTAIN_CAR_CONTINUOUS): the search steps MountainCar-v0 (gym 0.17-0.19 mountain_car.py)
                                   instead of CartPole-v0.  Hidden state (position, velocity), network input (float)position,
                                   (float)velocity; actions 0 (push left), 1 (none), 2 (push right); Node.r is the env's reward, -1.0;
                                   an episode ends at the goal.  The tree holds 128-byte three-action rows, so max_rollouts <= 16382.
                                   Every schedule and every other flag apply, except the trees-in-shared-memory whole-search kernel
                                   (thin batches run the two-phase kernel).  Hidden-state arrays (search roots, d_env_state, the dump's
                                   state, azg_env_step) are 2 wide; results and dump arrays carry 3 actions.  The reward model
                                   (azg_set_reward_model) stays the identity. */
#define AZG_FLAG_ENV_ACROBOT 64u /* discrete variant only, with num_actions 3 and state_dim 6 (not with either MountainCar flag): the
                                   search steps Acrobot-v1 (gym 0.17-0.19 acrobot.py: book dynamics, RK4 over dt = 0.2, no torque
                                   noise) instead of CartPole-v0.  Hidden state (theta1, theta2, dtheta1, dtheta2); network input the
                                   observation (float)cos theta1, sin theta1, cos theta2, sin theta2, dtheta1, dtheta2; actions 0, 1, 2
                                   (torque -1, 0, +1); Node.r is the env's reward, -1.0 before the goal and 0.0 at it; an episode ends
                                   at the goal.  gym's wrap loop is capped: a search or env step that reaches the cap fails with
                                   AZG_EWRAP.  The tree holds 128-byte three-action rows, so max_rollouts <= 16382.  Every schedule and
                                   every other flag apply, except the trees-in-shared-memory whole-search kernel (thin batches run the
                                   two-phase kernel).  Hidden-state arrays (search roots, d_env_state, the dump's state, azg_env_step)
                                   are 4 wide; observations (azg_env_step's d_obs, the self-play d_obs) are 6 wide; results and dump
                                   arrays carry 3 actions.  The reward model (azg_set_reward_model) stays the identity. */

typedef struct azg_engine azg_engine;

int azg_create(const azg_config* cfg, azg_engine** out);
void azg_destroy(azg_engine* e);
const char* azg_last_error(void);
const char* azg_version(void);

/* Network weights: flat f32 in state_dict order -- trunk.{0,2,..}.{weight,bias}, value_head.{weight,bias},
 * dist_head.{weight,bias} (policies.py:101-120, :255-259, :434, :588).  `flat` may be a host or a device
 * pointer (detected).  Replaces the per-node model.predict_V / predict_pi / sample_action callbacks
 * (mcts.py:406-416, :619-623, :652). */
int64_t azg_num_weights(const azg_engine* e);
int azg_set_weights(azg_engine* e, const float* flat, int64_t n, void* stream);

/* Batched MCTSDiscrete.search (mcts.py:418-462) over B CartPole (or MountainCar-v0, Acrobot-v1) roots.
 * d_root_state [B][4] f64 hidden env state (x, x_dot, theta, theta_dot); MountainCar [B][2] (position, velocity); Acrobot [B][4]
 * (theta1, theta2, dtheta1, dtheta2);
 * d_root_n_init [B] carried-over root visit count after forward() (mcts.py:495-526) or NULL;
 * tree_id0: global id of tree 0 -- tree i's RNG streams are keyed by tree_id0+i, which makes results
 * independent of batch composition and of how trees are sharded over GPUs. */
int azg_search_discrete(azg_engine* e, int32_t B, const double* d_root_state, const int32_t* d_root_n_init,
                        int32_t n_rollouts, int64_t tree_id0, void* stream);

/* Batched MCTSContinuous.search (mcts.py:656-702) over B Pendulum roots; d_root_state [B][2] (th, thdot)
 * (MountainCarContinuous: (position, velocity)). */
int azg_search_continuous(azg_engine* e, int32_t B, const double* d_root_state, int32_t n_rollouts, int64_t tree_id0,
                          void* stream);

/* MCTS.return_results (mcts.py:269-307) for the last search: per tree, root children in insertion order.
 * Row stride is azg_cmax(e).  actions: action index (discrete) or sampled action (continuous). */
int32_t azg_cmax(const azg_engine* e);
int azg_root_results(azg_engine* e, int32_t B, float* d_actions, int32_t* d_counts, double* d_Q, double* d_V_target,
                     int32_t* d_n_children, void* stream);

/* Host-buffer convenience = what MCTS*.search + return_results cost end to end: H2D of the roots,
 * search, result extraction, D2H of the results, synchronised on return.  h_root_n_init may be NULL
 * (and must be for the continuous variant). */
int azg_search_host(azg_engine* e, int32_t B, const double* h_root_state, const int32_t* h_root_n_init, int32_t n_rollouts,
                    int64_t tree_id0, float* h_actions, int32_t* h_counts, double* h_Q, double* h_V_target,
                    int32_t* h_n_children);

/* The same, pipelined: begin(slot) enqueues everything -- H2D of the roots, the search, result extraction and, on a copy stream, the D2H
 * of the results -- and returns at once; end(slot) blocks until that slot's results are in the caller's buffers and returns the search's
 * status.  Two slots (0, 1): with both in flight the PCIe transfer of one search's results runs under the next search.  All host
 * buffers must be page-locked and must stay untouched until end(slot). */
int azg_search_host_begin(azg_engine* e, int32_t slot, int32_t B, const double* h_root_state, const int32_t* h_root_n_init,
                          int32_t n_rollouts, int64_t tree_id0, float* h_actions, int32_t* h_counts, double* h_Q, double* h_V_target,
                          int32_t* h_n_children);
int azg_search_host_end(azg_engine* e, int32_t slot);

/* Device status of the last search(es), self-play steps and env steps: AZG_OK, AZG_ENAN, AZG_ECAPACITY or AZG_EWRAP.  Synchronises
 * `stream`. */
int azg_status(azg_engine* e, void* stream);

/* Re-key the Philox streams (tie-break / eps-greedy / action noise / self-play draws).  Stream-ordered: searches enqueued
 * after the call use the new key, also when they replay a captured CUDA graph.  The reference seeds once per run
 * (run_continuous.py:24-25, run_discrete.py:27-28). */
int azg_set_seed(azg_engine* e, uint64_t seed, void* stream);

/* Reward wrappers of the reference around the CartPole env the discrete search steps (rl/wrappers.py:58-105, selected by the
 * -v0r / -v0s / -v0rs name suffixes, rl/make_game.py:71-83).  They only change the reward a node is created with (mcts.py:449), and
 * for CartPole that is a constant per terminal flag: reward_step / reward_terminal = 1.0 / 1.0 without wrappers, 0.005 / -1 with
 * ReparametrizeWrapper, each / 250.0 with ScaleRewardWrapper (the host computes the constants with the wrappers' own Python
 * expressions).  Takes effect for searches enqueued after the call (synchronises the device and drops captured graphs when something
 * changes).  Not implemented, and refused by the drop-in classes: NormalizeWrapper (sklearn scaler), PILCOWrapper (scipy pdf),
 * ScaleRewardWrapper around Pendulum (it returns np.float32, whose promotion through the backup depends on the numpy version).  An
 * engine for any other env (the continuous ones, MountainCar-v0) accepts only the identity (1.0, 1.0). */
int azg_set_reward_model(azg_engine* e, double reward_step, double reward_terminal);

/* ---- self-play step (SURVEY 8f rank 1; BASELINE config 5) -------------------------------------------------------------
 * One environment step of B independent self-play environments, the body of the reference's episode loop
 * (run_continuous.py:117-142, run_discrete.py:100-122), batched and entirely on the device:
 *   re-key (key = azg_selfplay_seed(base_seed, step_index)) -> search from d_env_state -> root results, written to the
 *   replay-row buffers (buffer.store((s, actions, counts, Qs, V)), buffers.py:61) -> final action:
 *     continuous  actions[counts.argmax()] (agents.py:533; by_value: Qs.argmax());
 *     discrete    pi = stable_normalizer(counts | Qs, temperature) (helpers.py:9-27), pi.argmax() if deterministic else a
 *                 draw with np.random.choice's inverse-CDF rule (agents.py:294-301);
 *   -> the real Env.step -> if terminal or the episode reached max_episode_length: Env.reset() and a fresh tree
 *   (reset_mcts), else discrete tree reuse: d_root_n = visit count of the chosen child (mcts.py:495-526).
 * All pointers are device pointers owned by the caller; in/out arrays carry the state from step to step. */
typedef struct azg_selfplay_io {
    double* d_env_state;   /* in/out [B][4|2] hidden env state (CartPole x, x_dot, theta, theta_dot | Acrobot theta1, theta2, dtheta1, dtheta2 |
                              MountainCar position, velocity | Pendulum th, thdot |
                              MountainCarContinuous position, velocity) */
    int32_t* d_ep_step;    /* in/out [B] steps taken in the current episode */
    int32_t* d_episode;    /* in/out [B] episode counter (indexes the reset stream) */
    int32_t* d_root_n;     /* in/out [B] discrete only: root visit count carried into the next search; NULL for continuous */
    float* d_obs;          /* out [B][state_dim] observation the search started from (the replay row's s) */
    float* d_actions;      /* out [B][cmax] */
    int32_t* d_counts;     /* out [B][cmax] */
    double* d_Q;           /* out [B][cmax] */
    double* d_V_target;    /* out [B] */
    int32_t* d_n_children; /* out [B] */
    float* d_action_taken; /* out [B] */
    double* d_reward;      /* out [B] raw env reward of the real step */
    int32_t* d_done;       /* out [B] 1 if the episode ended with this step */
} azg_selfplay_io;

uint64_t azg_selfplay_seed(uint64_t base_seed, int64_t step_index);
int azg_selfplay_step(azg_engine* e, int32_t B, const azg_selfplay_io* io, int32_t n_rollouts, int64_t tree_id0,
                      int64_t step_index, uint64_t base_seed, int32_t max_episode_length, int32_t deterministic,
                      int32_t by_value, double temperature, void* stream);

/* ---- parity hooks (SURVEY 8b): evaluator injection and full tree dump -------------------------------- */
/* Tapes are device arrays indexed by tree and by node/row creation index, stride azg_rows(e):
 * V [B][R]; prior [B][R][A] (discrete); action [B][R] (continuous).  Passing d_V = NULL returns to the
 * engine's own MLP + noise.  With tapes set no network kernel runs. */
int32_t azg_rows(const azg_engine* e); /* = max_rollouts + 2 */
int azg_set_tapes(azg_engine* e, const float* d_V, const float* d_prior, const float* d_action);

typedef struct azg_dump_discrete { /* host arrays, R = azg_rows(e), A = num_actions; nodes in creation order */
    int32_t* n_nodes;  /* [B] */
    int32_t* parent;   /* [B][R] (-1 root) */
    int32_t* paction;  /* [B][R] */
    int32_t* node_n;   /* [B][R] Node.n */
    int32_t* terminal; /* [B][R] */
    float* V;          /* [B][R] */
    double* r;         /* [B][R] */
    double* state;     /* [B][R][4]; MountainCar [B][R][2] (Acrobot 4) */
    float* prior;      /* [B][R][A] */
    double* eW;        /* [B][R][A] Action.W */
    int32_t* en;       /* [B][R][A] Action.n */
    int32_t* echild;   /* [B][R][A] (-1 none) */
} azg_dump_discrete;

typedef struct azg_dump_continuous { /* host arrays; rows in creation order, row 0 = root */
    int32_t* n_rows;   /* [B] */
    int32_t* parent;   /* [B][R] (-1 root) */
    float* action;     /* [B][R] */
    double* eW;        /* [B][R] */
    int32_t* en;       /* [B][R] */
    int32_t* expanded; /* [B][R] */
    int32_t* node_n;   /* [B][R] */
    int32_t* terminal; /* [B][R] */
    float* V;          /* [B][R] */
    double* r;         /* [B][R] */
    double* state;     /* [B][R][2] */
    float* head;       /* [B][R][3K] mu, sigma, mixture prob */
} azg_dump_continuous;

int azg_dump_tree_discrete(azg_engine* e, int32_t B, const azg_dump_discrete* out);
int azg_dump_tree_continuous(azg_engine* e, int32_t B, const azg_dump_continuous* out);

/* counters of the last search, summed over trees: [0] simulations, [1] selection levels, [2] child edges
 * scanned, [3] progressive-widening inserts, [4] network evaluations, [5] RNG draws, [6] simulations that
 * ended on a terminal node, [7] kernels launched (or graph nodes replayed). */
int azg_get_counters(azg_engine* e, int32_t B, int64_t out[8]);

/* Cycle accounting of the whole-search kernel (AZG_FLAG_FUSED) since the last call, summed over CTAs, then reset (measured on
 * thread 0 of each CTA): out[0] kernel cycles, out[1] cycles in the tree phases (backup + select + expansion of every tree of the
 * CTA, up to the closing barrier), out[2] cycles waiting for the post-processing warps before a tree phase, out[4] CTAs counted,
 * out[5] which whole-search kernel the last search ran (1 two-phase, 2 warpgroups, 3 two-phase with the trees in shared memory).
 * Synchronises the device. */
int azg_fused_stats(azg_engine* e, int64_t out[8]);

/* Measurement hook: runs one search with direct launches, a CUDA-event pair around every kernel, and
 * returns total milliseconds and launch counts per kernel class: [0] tree step kernels (backup + select +
 * expansion/env step), [1] leaf evaluation (network), [2] setup (root init / root insert).  Synchronous. */
int azg_profile_search(azg_engine* e, int32_t B, const double* d_root_state, const int32_t* d_root_n_init,
                       int32_t n_rollouts, int64_t tree_id0, void* stream, float ms_out[3], int32_t launches_out[3]);

/* Batched network forward on its own (known-answer tests of the evaluation kernel):
 * d_x [n][state_dim] -> d_V [n], d_head [n][azg_head_dim(e)] post-processed head
 * (discrete: softmax priors [A]; continuous: mu[K], sigma[K], prob[K]). */
int32_t azg_head_dim(const azg_engine* e);
int azg_mlp_forward(azg_engine* e, int32_t n, const float* d_x, float* d_V, float* d_head, void* stream);

/* Batched env.step of the engine's env on its own (known-answer tests): d_state [n][4|2] (CartPole 4, MountainCar and the continuous
 * envs 2; Acrobot 4), d_action [n] (index as float for CartPole, MountainCar and Acrobot) -> d_next [n][4|2], d_reward [n] (raw env reward), d_terminal [n], d_obs [n][state_dim]. */
int azg_env_step(azg_engine* e, int32_t n, const double* d_state, const float* d_action, double* d_next, double* d_reward,
                 int32_t* d_terminal, float* d_obs, void* stream);

#ifdef __cplusplus
}
#endif
#endif

/*
 * azg_oracle.h -- CPU restatement of the alphazero-gym search hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is part of the product: only
 * tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
 * legs may load this library, and only as the checker / CPU baseline.  The CUDA
 * engine (alphazero_gym_b200/csrc) never includes or links anything from here.
 *
 * What is restated (reference = /root/reference, timoklein/alphazero-gym):
 *   alphazero/search/mcts.py:418-462   MCTSDiscrete.search
 *   alphazero/search/mcts.py:464-493   MCTSDiscrete.selectionUCT (PUCT)
 *   alphazero/search/mcts.py:385-416   MCTSDiscrete.evaluation
 *   alphazero/search/mcts.py:656-702   MCTSContinuous.search
 *   alphazero/search/mcts.py:704-741   MCTSContinuous.selectionUCT (PW + UCT)
 *   alphazero/search/mcts.py:602-654   add_value_estimate / add_pw_action
 *   alphazero/search/mcts.py:175-195   epsilon_greedy
 *   alphazero/search/mcts.py:241-267   backprop
 *   alphazero/search/mcts.py:269-307   return_results (+ value targets :91-173)
 *   alphazero/search/states.py:97-112  Action.update
 *   alphazero/search/states.py:252-275 NodeContinuous.check_pw
 *   alphazero/helpers.py:30-52         argmax with random tie-break
 *   alphazero/network/policies.py:154-160,275-352,436-458,590-631,656-669
 *                                      MLP trunk, value head, softmax / GMM head
 *   alphazero/network/distributions.py:50-63  bound*tanh(x)
 * Third-party arithmetic that is NOT under /root/reference (gym 0.17.2/0.19.0
 * classic_control CartPole-v0 / Pendulum-v0 / MountainCarContinuous-v0 /
 * MountainCar-v0 / Acrobot-v1 `step`) is restated from the published gym
 * source; see SURVEY.md section 8(c).  The config's `env` picks the env a
 * search steps; the search loops are the same for every env.
 *
 * Parity pinning: the reference has no tests or golden vectors.  This oracle is
 * pinned against outputs of the reference itself, generated in the build
 * container by oracle/gen_golden.py (imports /root/reference unmodified) and
 * committed under tests/golden/.  tests/test_oracle_vs_golden.py checks it.
 */
#ifndef AZG_ORACLE_H
#define AZG_ORACLE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AZO_DISCRETE 0
#define AZO_CONTINUOUS 1

#define AZO_ACT_RELU 0
#define AZO_ACT_ELU 1
#define AZO_ACT_LEAKYRELU 2 /* nn.LeakyReLU(): x > 0 ? x : 0.01 x   (network/utils.py:5-14) */
#define AZO_ACT_RELU6 3     /* nn.ReLU6(): min(max(x, 0), 6) */
#define AZO_ACT_SILU 4      /* nn.SiLU() ("swish" / "silu"): x / (1 + exp(-x)) */
#define AZO_ACT_HARDSWISH 5 /* nn.Hardswish(): x * min(max(x + 3, 0), 6) / 6 */

#define AZO_MATH_LIBM 0 /* glibc sin/cos/expf/... : what the python reference calls */
#define AZO_MATH_DET 1  /* op-for-op deterministic functions shared (as a spec) with the CUDA engine */

#define AZO_EVAL_FP32 0 /* every layer in FP32 FMA, k ascending (csrc/mlp.cuh) */
#define AZO_EVAL_Q8 1   /* hidden x hidden layers as exact int8-sliced fixed-point products (csrc/qmlp.cuh; contract below) */

#define AZO_VT_OFF_POLICY 0
#define AZO_VT_ON_POLICY 1
#define AZO_VT_GREEDY 2

#define AZO_MAX_LAYERS 8
#define AZO_MAX_K 8
#define AZO_MAX_A 8

typedef struct {
    int32_t variant;       /* AZO_DISCRETE | AZO_CONTINUOUS */
    int32_t n_rollouts;
    int32_t num_actions;   /* discrete: A */
    int32_t num_components;/* continuous: K (1 = DiagonalNormalPolicy, >1 = DiagonalGMMPolicy) */
    int32_t state_dim;     /* network input (the env's observation): 4 CartPole, 3 Pendulum, 2 MountainCar(Continuous), 6 Acrobot */
    int32_t hidden;        /* hidden width (all layers equal) */
    int32_t n_hidden;      /* number of hidden layers */
    int32_t activation;    /* AZO_ACT_* */
    int32_t math_mode;     /* AZO_MATH_* */
    int32_t v_target;      /* AZO_VT_* */
    int32_t puct_f32;      /* 1: prior*c_uct rounded to f32 (numpy>=2, NEP 50); 0: f64 (numpy 1.x) */
    int32_t use_eval_tape; /* 1: V / priors / actions come from tapes (evaluator injected) */
    double c_uct, gamma, epsilon, c_pw, kappa;
    float action_bound, log_std_min, log_std_max;
    uint64_t seed;         /* Philox key */
    int32_t eval_mode;     /* AZO_EVAL_* */
    int32_t rng_mode;      /* 0: Philox streams (default); 1 (AZO_RNG_MT19937, discrete search only): CPython's generator, seeded
                              with seed + global tree id at the start of every search (azg_oracle.c "AZO_RNG_MT19937") */
    /* reward wrappers of rl/wrappers.py around the env the search steps (rl/make_game.py:71-83, name suffixes -v0r / -v0s / -v0rs):
     * CartPole: the reward of a step is a constant per terminal flag -- 1.0 / 1.0 plain, 0.005 / -1 with ReparametrizeWrapper (:78-105),
     * / 250.0 with ScaleRewardWrapper (:58-75).  (Pendulum's ScaleRewardWrapper returns np.float32, whose promotion through the backup
     * depends on the numpy version: not restated.) */
    double reward_step, reward_terminal; /* CartPole only: any other env requires 1.0 / 1.0 */
    int32_t env;           /* AZO_ENV_* */
} azo_config;
#define AZO_ENV_DEFAULT 0                 /* the variant's own env: CartPole-v0 (discrete) / Pendulum-v0 (continuous) */
#define AZO_ENV_MOUNTAIN_CAR_CONTINUOUS 1 /* continuous, state_dim 2 */
#define AZO_ENV_MOUNTAIN_CAR 2            /* discrete, num_actions 3, state_dim 2 */
#define AZO_ENV_ACROBOT 3                 /* discrete, num_actions 3, state_dim 6 */
/* hidden env state (the tree's state rows hold it; 4 doubles per discrete row, 2 per continuous row):
 *   CartPole x, xdot, th, thdot | Pendulum th, thdot | MountainCar(Continuous) position, velocity | Acrobot th1, th2, dth1, dth2 */

#define AZO_ERR_WRAP -4 /* Acrobot: an angle needed more than 64 iterations of a wrap loop (gym's loop is unbounded) */
#define AZO_RNG_PHILOX 0
#define AZO_RNG_MT19937 1

/* AZO_EVAL_Q8 contract (the arithmetic the tcgen05 kind::i8 kernel performs; every step is exact integer
 * arithmetic or one correctly rounded IEEE f32 operation, so CPU and GPU agree bit for bit):
 *   layer 0 (state_dim -> H): FP32 FMA as in AZO_EVAL_FP32.
 *   scaling: for a vector with largest magnitude vmax, e = clamp(biased_exponent(f32(vmax * 1.004f)), 32, 200) and
 *     q = rni_sat(v * 2^(149-e)), so |q| <= 8355711 and the balanced signed base-256 digits q = hi*2^16 + mid*2^8 + lo
 *     (bytes of (q + 0x8080) ^ 0x8080) all fit int8.
 *   weights of a hidden layer: one scale per output j (vmax over k);  cw[j] = 2^(e-133).
 *   activations: one scale per row (vmax over the H inputs of the layer);  cx = 2^(e-149).
 *   products (int32, exact):  PA = sum xh*wh;  PB = sum xh*wm + xm*wh;  PC = sum xh*wl + xm*wm + xl*wh
 *     (order-5/6 digit products dropped: relative weight <= 2^-24 of the leading product; measured error of V
 *     against an f64 evaluation is 2x that of the FP32 path, tests/test_q8_eval.py).
 *   y[j] = fma(fma(fma((f32)PA, 256, (f32)PB), 256, (f32)PC), cx * cw[j], bias[j]);  a'[j] = act(y[j]).
 *   heads: partial[q] = fma chain over k in [32q, 32q+32) from 0;  out = ((p0 + p1) + (p2 + p3)) + bias
 *     (for H = 128; in general H/32 partials summed pairwise left to right). */

/* Row counts: a search of N rollouts creates at most N+1 nodes (root + one per rollout);
 * the continuous tree can hold one extra unexpanded root edge (c_pw > 1), hence N+2 rows. */
static inline int azo_rows(const azo_config* c) { return c->n_rollouts + 2; }

/* ---- tree dump: logical layout shared with the engine's azg_dump_tree ------------ */
/* Discrete: per tree, nodes in creation order (node 0 = root), capacity R = azo_rows(). */
typedef struct {
    int32_t* n_nodes;   /* [B] */
    int32_t* parent;    /* [B][R]   parent node (-1 root) */
    int32_t* paction;   /* [B][R]   action taken at the parent */
    int32_t* node_n;    /* [B][R]   Node.n */
    int32_t* terminal;  /* [B][R] */
    float* V;           /* [B][R]   Node.V */
    double* r;          /* [B][R]   Node.r */
    double* state;      /* [B][R][HS] hidden env state: HS = 4 CartPole / Acrobot, 2 MountainCar */
    float* prior;       /* [B][R][A] */
    double* eW;         /* [B][R][A] Action.W */
    int32_t* en;        /* [B][R][A] Action.n */
    int32_t* echild;    /* [B][R][A] child node or -1 */
} azo_dump_discrete;

/* Continuous: per tree, rows in creation order; row 0 = root (no edge part), row i>0 is an
 * edge (ActionContinuous) plus, once expanded, the child node it leads to. */
typedef struct {
    int32_t* n_rows;    /* [B] */
    int32_t* parent;    /* [B][R]  parent row (-1 root) */
    float* action;      /* [B][R]  Action.action */
    double* eW;         /* [B][R]  Action.W */
    int32_t* en;        /* [B][R]  Action.n */
    int32_t* expanded;  /* [B][R]  1 once the child node exists */
    int32_t* node_n;    /* [B][R]  Node.n */
    int32_t* terminal;  /* [B][R] */
    float* V;           /* [B][R] */
    double* r;          /* [B][R]  (already divided by PENDULUM_R_SCALE) */
    double* state;      /* [B][R][2] hidden env state */
    float* head;        /* [B][R][3K] cached policy head: mu[K], sigma[K], prob[K] */
} azo_dump_continuous;

/* root results (mcts.py:269-307): Cmax columns, insertion order */
typedef struct {
    int32_t cmax;
    int32_t* n_children; /* [B] */
    float* actions;      /* [B][Cmax] (discrete: the action index as float) */
    int32_t* counts;     /* [B][Cmax] */
    double* Q;           /* [B][Cmax] */
    double* V_target;    /* [B] */
    int64_t* counters;   /* [8]: sims, levels, children scanned, pw inserts, evals, rng draws, terminal leaves, reserved */
} azo_results;

/* tapes (evaluator injection, SURVEY 8c parity level A); any pointer may be NULL */
typedef struct {
    const float* V;      /* [B][R]    value of node/row i (creation order) */
    const float* prior;  /* [B][R][A] discrete */
    const float* action; /* [B][R]    continuous: action of row i */
} azo_tapes;

/* Run B independent searches.  weights: flat f32 in state_dict order
 * (trunk.{0,2,..}.{weight,bias}, value_head.{weight,bias}, dist_head.{weight,bias}).
 * root_state: [B][HS] hidden env states (HS: see AZO_ENV_*).
 * root_n_init: [B] carried-over root visit count (discrete tree reuse quirk) or NULL.
 * tree_id0: global id of tree 0 (Philox stream key).  dump_* may be NULL.
 * Returns 0, or <0 on error (-2 bad config, -3 NaN in UCT, AZO_ERR_WRAP). */
int azo_search(const azo_config* cfg, const float* weights, int64_t n_weights, int32_t B, const double* root_state,
               const int32_t* root_n_init, int64_t tree_id0, const azo_tapes* tapes, azo_results* res,
               azo_dump_discrete* dd, azo_dump_continuous* dc, int32_t n_threads);

int64_t azo_num_weights(const azo_config* cfg);
int32_t azo_head_dim(const azo_config* cfg);
int32_t azo_pw_limit(double c_pw, double kappa, int32_t n); /* ceil(c_pw*(n+1)**kappa), states.py:252-275 */

/* ---- building blocks exported for known-answer tests and the golden harness ------- */
uint32_t azo_rng_u32(uint64_t seed, int64_t tree, int32_t stream, int64_t idx, int32_t block, int32_t word);
/* noise for the j-th progressive-widening insert of `tree`: component uniform + K standard normals */
/* rng_block of n counters: out[i][0..3] = the four words of (tree[i], stream[i], idx[i], block[i]) */
void azo_rng_block_batch(uint64_t seed, const int64_t* tree, const int32_t* stream, const int64_t* idx, const int32_t* block, int64_t n,
                         uint32_t* out);
void azo_noise(uint64_t seed, int64_t tree, int64_t j, int32_t K, float* u_comp, float* z);
/* batched MLP forward (deterministic fmaf order): out_V [n], out_head [n][P] raw head outputs */
void azo_mlp_forward(const azo_config* cfg, const float* weights, int32_t n, const float* x, float* out_V, float* out_head);
/* head post-processing: discrete softmax priors [A]; continuous (mu,sigma,prob)[3K] */
void azo_head_post(const azo_config* cfg, const float* raw, float* out);
float azo_sample_action(const azo_config* cfg, const float* head, float u_comp, const float* z);
/* one env step of the config's env (discrete: the action index as float); returns terminal, or AZO_ERR_WRAP */
int azo_env_step(const azo_config* cfg, const double* s_in, float action, double* s_out, double* reward, float* obs);
void azo_obs(const azo_config* cfg, const double* s, float* obs); /* observation of a hidden env state */

float azo_det_expf(float x);
float azo_det_expm1f(float x);
float azo_det_tanhf(float x);
double azo_det_sin(double x);
double azo_det_cos(double x);
double azo_det_log(double x);

/* Batched evaluation of one deterministic function over n elements with n_threads threads (exhaustive accuracy sweeps
 * and engine comparisons run at C speed).  fn = AZO_FN_*: expf / expm1f / tanhf and AZO_FN_ACT + AZO_ACT_* (act_fn in
 * AZO_MATH_DET mode) read and write float; sin / cos / log read and write double. */
#define AZO_FN_EXPF 0
#define AZO_FN_EXPM1F 1
#define AZO_FN_TANHF 2
#define AZO_FN_SIN 3
#define AZO_FN_COS 4
#define AZO_FN_LOG 5
#define AZO_FN_ACT 16
int azo_det_eval(int32_t fn, const void* in, void* out, int64_t n, int32_t n_threads);

/* The MT19937 generators of AZO_RNG_MT19937 on a caller-held state of 625 words (624 state words + the index word).
 * CPython `random`: azo_mt_seed = random.seed(int) (init_by_array), azo_mt_u32 = getrandbits(32), azo_mt_random =
 * random(), azo_mt_below(n) = _randbelow(n).  torch's CPU generator: azo_torch_seed = torch.manual_seed (init_genrand of the
 * low 32 bits), azo_torch_uniform = one double uniform (53 bits of two outputs). */
void azo_mt_seed(uint32_t* st, uint64_t seed);
uint32_t azo_mt_u32(uint32_t* st);
double azo_mt_random(uint32_t* st);
int32_t azo_mt_below(uint32_t* st, int32_t n);
void azo_torch_seed(uint32_t* st, uint64_t seed);
double azo_torch_uniform(uint32_t* st);

#ifdef __cplusplus
}
#endif
#endif

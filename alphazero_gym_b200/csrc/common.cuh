// common.cuh -- table layouts, kernel parameter block and Philox for the batched MCTS engine (sm_100a).
//
// Data layout in HBM (DESIGN.md section 3).  Trees are independent; everything is indexed tree-major
// (tree t owns rows [t*R, (t+1)*R), R = max_rollouts + 2).  The reference's pointer-linked
// Node / Action objects (alphazero/search/states.py:8-112) become:
//   * one packed HOT row per node, sized to DRAM sectors so a random node visit costs whole sectors
//     only: 64 B for the discrete tree (node + its A=2 edges) and 64 B for the continuous tree (sector 0:
//     edge statistics + the child node it leads to -- edges and non-root nodes are 1:1, SURVEY 7-4;
//     sector 1: that node's inline child list).  64 B is also the DRAM burst, so a row miss wastes nothing;
//   * the continuous tree adds a 64 B control block per tree (scalars, inline path, root child map) and a root edge table (the
//     root's children statistics, 32 B each), both TREE-INTERLEAVED ([4][trees] chunk planes / [16][trees], see TreeParams);
//   * COLD structure-of-arrays side tables that select/backup never touch: CartPole env state, cached policy head.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#define AZG_MAX_K 8
#define AZG_PENDULUM_R_SCALE 16.2736044 /* mcts.py:20 */
#define AZG_TAB 1024

// ---- hot rows ----------------------------------------------------------------------------------
struct __align__(16) DRow {  // NodeDiscrete + its ActionDiscrete[2]   (states.py:115-191, :292-362)
    double W[2];             // Action.W
    double r;                // Node.r
    int32_t n_e[2];          // Action.n
    float prior[2];          // Node.priors
    float V;                 // Node.V (0 for terminal nodes, mcts.py:406-410)
    int32_t node_n;          // Node.n
    uint16_t child[2];       // Action.child_node (DROW_NONE if absent)
    uint16_t parent;         // Node.parent_action.parent_node
    uint8_t paction;         // Node.parent_action.action
    uint8_t flags;           // ROW_TERMINAL
    uint32_t pad[2];
};
static_assert(sizeof(DRow) == 64, "discrete row must be two 32 B sectors");
#define DROW_NONE 0xFFFFu

// The three-action row (MountainCar-v0): two aligned 64 B lines.  Line 0 holds everything the descent reads at a node, so a level
// still costs one 64 B burst; line 1 holds what only the backup (r) and the tree dump (parent links) read.
struct __align__(16) D3Row {  // NodeDiscrete + its ActionDiscrete[3]
    // line 0
    double W[3];             // Action.W
    int32_t n_e[3];          // Action.n
    float prior[3];          // Node.priors
    float V;                 // Node.V (0 for terminal nodes)
    int32_t node_n;          // Node.n
    uint16_t child[3];       // Action.child_node (DROW_NONE if absent)
    uint8_t flags;           // ROW_TERMINAL
    uint8_t pad0;
    // line 1
    double r;                // Node.r
    uint16_t parent;         // Node.parent_action.parent_node
    uint8_t paction;         // Node.parent_action.action
    uint8_t pad1[53];
};
static_assert(sizeof(D3Row) == 128, "three-action row must be two 64 B lines");
static_assert(offsetof(D3Row, n_e) == 24 && offsetof(D3Row, prior) == 36 && offsetof(D3Row, V) == 48 && offsetof(D3Row, node_n) == 52 &&
              offsetof(D3Row, child) == 56 && offsetof(D3Row, flags) == 62 && offsetof(D3Row, r) == 64, "line 0 = what the descent reads");

struct __align__(16) CRow {  // ActionContinuous + the NodeContinuous it leads to (states.py:194-289, :365-433)
    // sector 0 ("hot" sector, struct CHot) -- read for every child scanned by UCT and rewritten by backup.
    // For children of the ROOT this sector is not used: their hot sectors live contiguously in the root edge
    // table (TreeParams::et), because the root is scanned in every simulation and has up to 16 children.
    // first 16 bytes = everything the UCT scan reads (one LDG.128 per child) and everything backup writes (one STG.128)
    double W;                // Action.W
    int32_t n_e;             // Action.n
    uint32_t nn_flags;       // child Node.n in bits 0..23 | CROW_EXPANDED | CROW_TERMINAL
    double r;                // child Node.r (already / PENDULUM_R_SCALE)
    float V;                 // child Node.V
    float action;            // Action.action
    // sector 1 -- the child node's own child_actions list (insertion order) and its hidden env state; read
    // only when the descent enters this node, appended to by progressive widening
    uint8_t kids[15];        // row indices
    uint8_t nkids;
    double th, thdot;        // Pendulum hidden state of the node
};
static_assert(sizeof(CRow) == 64, "continuous row must be two 32 B sectors (one 64 B DRAM burst)");
#define CROW_MAX_KIDS 15
#define CROOT_MAX_KIDS 16
#define ROW_TERMINAL 1u
#define CROW_NMASK 0x00FFFFFFu
#define CROW_EXPANDED 0x01000000u
#define CROW_TERMINAL 0x02000000u

struct __align__(16) CHot {  // sector 0 of a CRow / one entry of the root edge table
    double W;
    int32_t n_e;
    uint32_t nn_flags;
    double r;
    float V, action;
};
static_assert(offsetof(CHot, n_e) == 8 && offsetof(CHot, r) == 16 && offsetof(CRow, r) == 16 && offsetof(CRow, kids) == 32, "hot sector layout");
static_assert(sizeof(CHot) == 32, "hot sector");

struct __align__(16) CCtl {  // per-tree control block: everything a simulation needs besides rows, in ONE 64 B line
    uint8_t n_rows, depth, root_nk, j0;  // rows in use, recorded path length, root children, root-edge index of path[0]
    int32_t draws;           // selection RNG draw counter (stream 0)
    int32_t leaf;            // LEAF_* word for the evaluation kernel
    int32_t root_nn;         // root Node.n
    float root_V;            // root Node.V
    uint16_t pw;             // progressive-widening insert counter (stream 1 index)
    uint16_t pad;
    double leafR;            // return at the leaf edge of the current simulation: r + gamma*V
    uint8_t path[16];        // rows visited by the current simulation (deeper levels spill to TreeParams::path)
    uint8_t root_kids[16];   // row index of root child j (insertion order)
};
static_assert(sizeof(CCtl) == 64, "control block must be one 64 B line");

// leaf word handed from the tree kernels to the evaluation kernel
#define LEAF_ROW_MASK 0xFFFF
#define LEAF_J_SHIFT 16              // continuous: index of the leaf in the root edge table ...
#define LEAF_ROOTCHILD (1 << 28)     // ... valid when the leaf is a child of the root
#define LEAF_EVAL (1 << 29)      // the leaf is new: evaluate it
#define LEAF_TERMINAL (1 << 30)  // V is forced to 0

#define ERR_NAN 1
#define ERR_CAPACITY 2
#define ERR_WRAP 4  // Acrobot: an angle reached ACROBOT_WRAP_CAP iterations of wrap (env.cuh)

struct TreeParams {
    int32_t B, R, A, K, HS;  // trees, rows per tree, actions, mixture components, head stride (floats)
    int32_t puct_f32, v_target, use_tape;
    double c_uct, gamma, epsilon;
    double reward_step, reward_terminal;  // CartPole reward of a step / of the terminating step (1.0 / 1.0; rl/wrappers.py -> azg_set_reward_model)
    float gamma_f32, action_bound;
    const uint64_t* seedp;  // Philox key, read from device memory so that azg_set_seed re-keys a captured graph
    int64_t tree_id0;
    int32_t tree_word;      // launches captured into a CUDA graph: the global id of tree 0 is seedp[1] (and tree_id0 is 0), so that one
                            // graph serves every tree_id0 (the drop-in classes search with a new id every call)
    // discrete tables
    DRow* drows;      // [B][R]  (MountainCar-v0, Acrobot-v1: D3Row [B][R], same pointer)
    double* dstate;   // [B][R][4]  (MountainCar-v0: the first 2 of each 4; Acrobot-v1: all 4)
    // continuous tables
    CRow* crows;      // [B][R]
    float* chead;     // [B][R][HS]  mu[K], sigma[K], prob[K]
    // Tree-INTERLEAVED tables (BS = max_trees is the stride): a warp advances 32 consecutive trees in lockstep, so entry j of tree t
    // sits next to entry j of tree t + 1 and a warp-wide access touches 4 (control chunk) or 8 (edge) lines instead of 32 --
    // the tree kernels are bound by L1 tag lookups of per-thread scattered accesses, not by HBM (profiles/README.md r1f)
    CHot* et;         // [16][BS]  root edge table: hot sectors of the root's children, insertion order; child j of tree t = et[j * BS + t]
    uint4* ctl;       // [4][BS]   control blocks (CCtl) as four 16-byte chunk planes: chunk k of tree t = ctl[k * BS + t]
    int32_t BS;
    const int32_t* pw_table;  // [max_rollouts + 2]  ceil(c_pw * (n+1)^kappa), built on the host
    const double* rcp_tab;    // [AZG_TAB + 1]  1.0 / i  (host-built, correctly rounded), see div_small
    const double* sqrt_tab;   // [AZG_TAB + 1]  sqrt(i)
    // per-tree scalars
    // per-tree scalars of the discrete tree (the continuous tree keeps them in CCtl)
    int32_t* n_rows;  // rows / nodes in use
    int32_t* draws;   // selection RNG draw counter (stream 0)
    int32_t* leaf;    // LEAF_* word
    uint8_t* path;    // [B][R] continuous: path entries beyond the 16 held in CCtl
    uint32_t* mt;     // [B][625] AZG_FLAG_RNG_MT19937: per-tree MT19937 state + index word of CPython's generator (see mt19937 below)
    uint32_t* tmt;    // [B][628] AZG_FLAG_RNG_MT19937, continuous: torch's CPU generator (state, index, cached normal lo / hi / valid)
    int32_t rng_mt;
    uint16_t* dpath;  // [B][R] discrete: the current simulation's path, (row << 1 | action) per level (three actions: row << 2 | action),
                      // root first (read by the backup)
    int32_t* ddepth;  // [B]    discrete: its length
    uint32_t* ctr;    // [4][B]: levels, children scanned, terminal-leaf sims, evals
    float4* X;        // [B][XW] network input of the leaf (XW = 2 for Acrobot's 6 inputs, 1 otherwise)
    const double* root_state;
    const int32_t* root_n_init;
    int32_t* err;
    unsigned long long* prof;  // AZG_TREE_PROF builds: cycle accounting of the tree step per section (warp time, lane 0)
    // evaluator injection (parity level A)
    const float* tapeV;
    const float* tapeP;
    const float* tapeA;
};

#ifdef AZG_TREE_PROF
#define TP_BEGIN() long long tp_last = clock64()
#define TP_STAMP(k) do { const long long _t = clock64(); if ((threadIdx.x & 31) == 0 && p.prof) atomicAdd(p.prof + (k), (unsigned long long)(_t - tp_last)); tp_last = _t; } while (0)
#else
#define TP_BEGIN()
#define TP_STAMP(k)
#endif

// ---- IEEE division by a small integer without the division routine ------------------------------------------------
// Q = W / n and sqrt(N + 1) / (n + 1) sit on the select chain between two dependent loads, and DDIV / DSQRT are ~40-instruction
// dependent sequences.  With y = RN(1 / b) from a table: q = RN(a y), r = a - q b (exact in one fma), RN(q + r y) is the
// correctly rounded quotient a / b (Markstein's final division step; b is a small integer, so the one exceptional divisor
// pattern, an all-ones significand, cannot occur; 4e8 random cases checked against a / b on the CPU).  Zero, subnormal-range
// and non-finite numerators take the ordinary division.
__device__ __forceinline__ double div_small(double a, int b, const double* rcp, int tab_n) {
    const double fa = fabs(a);
    if (b > tab_n || !(fa > 1e-250 && fa < 1e250)) return a / (double)b;
    const double y = rcp[b];  // plain load: the table may sit in shared memory (whole-search kernel)
    const double q = __dmul_rn(a, y);
    const double r = __fma_rn(-q, (double)b, a);
    return __fma_rn(r, y, q);
}
__device__ __forceinline__ double sqrt_small(int n, const double* tab, int tab_n) {
    return n <= tab_n ? tab[n] : sqrt((double)n);
}
// The three small lookup tables of the select step.  k_step_* read them from global memory (L1-resident there); the whole-search
// kernel, whose L1 is a few KB next to 215 KB of shared memory, keeps the first FUSED_TAB + 1 entries in shared memory
// (continuous trees hold at most 255 rows, so visit counts + 1 stay below 256).
#define FUSED_TAB 255
struct Tabs {
    const int32_t* pw;   // progressive-widening limits
    const double* rcp;   // 1 / i
    const double* sq;    // sqrt(i)
    int n;               // largest index held
};

// ---- Philox4x32-10 (Salmon et al. SC'11); counter layout documented in DESIGN.md section 5 ---------
struct u32x4 { uint32_t x, y, z, w; };

__device__ __forceinline__ u32x4 philox4x32_10(u32x4 c, uint32_t k0, uint32_t k1) {
#pragma unroll 1  // rolled: the generator is inlined at half a dozen call sites of the tree kernels and never on a throughput path
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        u32x4 n;
        n.x = hi1 ^ c.y ^ k0;
        n.y = lo1;
        n.z = hi0 ^ c.w ^ k1;
        n.w = lo0;
        c = n;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return c;
}

__device__ __forceinline__ u32x4 rng_block(uint64_t seed, int64_t tree, int stream, int64_t idx, int block) {
    u32x4 c;
    c.x = (uint32_t)idx;
    c.y = (uint32_t)((uint64_t)idx >> 32) ^ ((uint32_t)block << 16);
    c.z = (uint32_t)tree;
    c.w = (uint32_t)((uint64_t)tree >> 32) ^ ((uint32_t)stream << 24);
    return philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
}

// four selection draws at once (.x of the blocks of draw indices idx0, idx0 + stride, ...): the four Philox chains are
// independent, so they interleave in the pipeline and cost about the latency of one
__device__ __forceinline__ void rng_select_u32x4(uint64_t seed, int64_t tree, int idx0, int stride, uint32_t out[4]) {
    uint32_t cx[4], cy[4], cz[4], cw[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int64_t idx = idx0 + q * stride;
        cx[q] = (uint32_t)idx;
        cy[q] = (uint32_t)((uint64_t)idx >> 32);
        cz[q] = (uint32_t)tree;
        cw[q] = (uint32_t)((uint64_t)tree >> 32);  // stream 0, block 0
    }
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll 1
    for (int r = 0; r < 10; ++r) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const uint32_t hi0 = __umulhi(0xD2511F53u, cx[q]), lo0 = 0xD2511F53u * cx[q];
            const uint32_t hi1 = __umulhi(0xCD9E8D57u, cz[q]), lo1 = 0xCD9E8D57u * cz[q];
            cx[q] = hi1 ^ cy[q] ^ k0;
            cy[q] = lo1;
            cz[q] = hi0 ^ cw[q] ^ k1;
            cw[q] = lo0;
        }
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) out[q] = cx[q];
}

// ---- AZG_FLAG_RNG_MT19937 (SURVEY 8f rank 4): CPython's generator for the selection draws of the discrete search, so that an
// UN-SHIMMED reference run (stock `random` module, random.seed(seed + tree) right before MCTSDiscrete.search) is reproduced bit for
// bit: init_by_array seeding (CPython random_seed with an int), random() = 53 bits of two outputs, choice / randint =
// _randbelow_with_getrandbits (k = n.bit_length(); take the top k bits until < n).  Same contract as oracle/azg_oracle.c
// "AZO_RNG_MT19937"; a compatibility mode, not a fast path (2.5 KB of state per tree in HBM).
#define MT_N 624
__device__ __forceinline__ void mt_seed_dev(uint32_t* mt, uint64_t seed) {
    const uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    const int klen = key[1] ? 2 : 1;
    mt[0] = 19650218u;
    for (int i = 1; i < MT_N; ++i) mt[i] = 1812433253u * (mt[i - 1] ^ (mt[i - 1] >> 30)) + (uint32_t)i;
    int i = 1, j = 0;
    for (int k = MT_N; k; --k) {
        mt[i] = (mt[i] ^ ((mt[i - 1] ^ (mt[i - 1] >> 30)) * 1664525u)) + key[j] + (uint32_t)j;
        ++i; ++j;
        if (i >= MT_N) { mt[0] = mt[MT_N - 1]; i = 1; }
        if (j >= klen) j = 0;
    }
    for (int k = MT_N - 1; k; --k) {
        mt[i] = (mt[i] ^ ((mt[i - 1] ^ (mt[i - 1] >> 30)) * 1566083941u)) - (uint32_t)i;
        ++i;
        if (i >= MT_N) { mt[0] = mt[MT_N - 1]; i = 1; }
    }
    mt[0] = 0x80000000u;
    mt[MT_N] = MT_N;  // index word: the first output regenerates the state
}
__device__ __forceinline__ uint32_t mt_next_dev(uint32_t* mt, int& mti, int& draws) {
    if (mti >= MT_N) {
        int kk;
        uint32_t y;
        for (kk = 0; kk < MT_N - 397; ++kk) { y = (mt[kk] & 0x80000000u) | (mt[kk + 1] & 0x7fffffffu); mt[kk] = mt[kk + 397] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u); }
        for (; kk < MT_N - 1; ++kk) { y = (mt[kk] & 0x80000000u) | (mt[kk + 1] & 0x7fffffffu); mt[kk] = mt[kk + (397 - MT_N)] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u); }
        y = (mt[MT_N - 1] & 0x80000000u) | (mt[0] & 0x7fffffffu);
        mt[MT_N - 1] = mt[396] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
        mti = 0;
    }
    uint32_t y = mt[mti++];
    y ^= y >> 11; y ^= (y << 7) & 0x9d2c5680u; y ^= (y << 15) & 0xefc60000u; y ^= y >> 18;
    ++draws;
    return y;
}
__device__ __forceinline__ double mt_random_dev(uint32_t* mt, int& mti, int& draws) {  // random.random()
    const uint32_t a = mt_next_dev(mt, mti, draws) >> 5, b = mt_next_dev(mt, mti, draws) >> 6;
    return ((double)a * 67108864.0 + (double)b) * (1.0 / 9007199254740992.0);
}
__device__ __forceinline__ int mt_below_dev(uint32_t* mt, int& mti, int& draws, int n) {  // random.choice over n items / randint(0, n - 1)
    const int k = 32 - __clz(n);  // n.bit_length()
    uint32_t r = mt_next_dev(mt, mti, draws) >> (32 - k);
    while ((int)r >= n) r = mt_next_dev(mt, mti, draws) >> (32 - k);
    return (int)r;
}

// global id of the launch's tree 0 (keys every random stream)
__device__ __forceinline__ int64_t tree_base(const TreeParams& p) { return p.tree_id0 + (p.tree_word ? (int64_t)__ldg(p.seedp + 1) : 0); }

// ---- AZG_FLAG_RNG_MT19937, continuous search: torch's global CPU generator for the action noise, exactly as an UN-WRAPPED
// `model.sample_action` consumes it after torch.manual_seed(seed + tree) (contract and derivation: oracle/azg_oracle.c
// torch_sample_action): at::mt19937 seeded by init_genrand; uniform = 53 bits of (out1 << 32 | out2); torch.multinomial(probs, 1) =
// argmax_k probs_k / (float)(-log1p(-uniform)); normal = Box-Muller on doubles with the sine kept for the next call.
#define TMT_WORDS (MT_N + 4)  // state, index, cached normal (lo, hi), cache-valid flag
__device__ __forceinline__ void tmt_seed_dev(uint32_t* mt, uint64_t seed) {
    mt[0] = (uint32_t)seed;
    for (int i = 1; i < MT_N; ++i) mt[i] = 1812433253u * (mt[i - 1] ^ (mt[i - 1] >> 30)) + (uint32_t)i;
    mt[MT_N] = MT_N;
    mt[MT_N + 1] = mt[MT_N + 2] = mt[MT_N + 3] = 0;
}
__device__ __forceinline__ double tmt_uniform_dev(uint32_t* mt, int& mti) {
    int dummy = 0;
    const uint64_t hi = mt_next_dev(mt, mti, dummy), lo = mt_next_dev(mt, mti, dummy);
    return (double)(((hi << 32) | lo) & ((1ull << 53) - 1)) * (1.0 / 9007199254740992.0);
}

// stream 0: random.random() / random.choice / random.randint replacements (helpers.py:51, mcts.py:190-192)
__device__ __forceinline__ uint32_t rng_select_u32(const TreeParams& p, int64_t tree, int draw) {
    return rng_block(__ldg(p.seedp), tree, 0, draw, 0).x;
}
__device__ __forceinline__ float u32_to_unit(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-08f; }
__device__ __forceinline__ int u32_to_index(uint32_t x, int n) { return (int)__umulhi(x, (uint32_t)n); }

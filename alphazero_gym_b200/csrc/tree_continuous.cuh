// tree_continuous.cuh -- backup + progressive-widening / UCT select + expansion for the continuous tree.
//
// Reference: MCTSContinuous.search (mcts.py:656-702), selectionUCT (:704-741), add_pw_action (:625-654),
// NodeContinuous.check_pw (states.py:252-275), epsilon_greedy (mcts.py:175-195), helpers.argmax
// (helpers.py:30-52), MCTS.backprop (mcts.py:241-267), DiagonalGMMPolicy.sample_action
// (policies.py:656-669) with SquashedNormal (distributions.py:50-63, :205-245).
//
// Mapping: ONE THREAD PER TREE, a warp advances 32 trees in lockstep.  The first version of this kernel
// gave each tree a 16-lane sub-warp with shuffle arg-max over children gathered one per lane; ncu showed
// it issue-bound (every lane re-executes the scalar control flow: ~480 warp instructions per simulated
// tree, profiles/r1a_ncu_step.csv) and barrier-bound on its dense f64 phases.  With a thread per tree the
// same work costs ~1/10 of the issue slots, the f64 env step / Box-Muller run on full warps with no
// barriers, and memory-level parallelism comes from 65536 independent threads instead of from lanes.
//
// What bounds the step (profiles/README.md r1f, DESIGN.md 4.1): a chain of dependent loads per tree (17 us floor at any batch size)
// plus, beyond ~200 trees per SM, the L1 tag lookups of per-thread scattered accesses -- not HBM bandwidth.  Hence the layout:
//   * one 64 B control block per tree (CCtl: every scalar, the recorded path, the root's child map) stored as four 16-byte chunk
//     planes [4][trees], and the root edge table (the statistics sectors of the root's children: the root is scanned in every
//     simulation and has the widest fan-out) as [16][trees]: a warp's 32 consecutive trees touch 4 / 8 lines per access, not 32;
//   * W, n and the child node's n in the first 16 bytes of a hot sector: one load per scanned child, one store per backup level;
//   * a node's hidden env state rides in the second sector of its row together with its child list, so entering a node and
//     expanding below it cost no extra line.
#pragma once
#include "common.cuh"
#include "env.cuh"

__device__ __forceinline__ CHot load_hot(const void* p) {
    CHot h;
    const uint4* s = reinterpret_cast<const uint4*>(p);
    uint4* d = reinterpret_cast<uint4*>(&h);
    d[0] = s[0]; d[1] = s[1];
    return h;
}
__device__ __forceinline__ void store_hot(void* p, const CHot& h) {
    const uint4* s = reinterpret_cast<const uint4*>(&h);
    uint4* d = reinterpret_cast<uint4*>(p);
    d[0] = s[0]; d[1] = s[1];
}
struct CSec1 {  // sector 1 of a CRow
    uint32_t kw[4];  // kids[15] + nkids in the top byte of kw[3]
    double th, thdot;
};
__device__ __forceinline__ CSec1 load_sec1(const CRow* p) {
    CSec1 s;
    const uint4* q = reinterpret_cast<const uint4*>(p);
    const uint4 a = q[2], b = q[3];
    s.kw[0] = a.x; s.kw[1] = a.y; s.kw[2] = a.z; s.kw[3] = a.w;
    s.th = __hiloint2double((int)b.y, (int)b.x);
    s.thdot = __hiloint2double((int)b.w, (int)b.z);
    return s;
}
__device__ __forceinline__ void store_sec1_new(CRow* p, double th, double thdot) {
    uint4* q = reinterpret_cast<uint4*>(p);
    q[2] = make_uint4(0, 0, 0, 0);
    q[3] = make_uint4((uint32_t)__double2loint(th), (uint32_t)__double2hiint(th), (uint32_t)__double2loint(thdot),
                      (uint32_t)__double2hiint(thdot));
}
// control block of tree t: four 16-byte chunks in four tree-interleaved planes (common.cuh)
__device__ __forceinline__ CCtl load_ctl(const uint4* ctl, int BS, int t) {
    CCtl c;
    uint4* d = reinterpret_cast<uint4*>(&c);
#pragma unroll
    for (int k = 0; k < 4; ++k) d[k] = ctl[(size_t)k * BS + t];
    return c;
}
__device__ __forceinline__ void store_ctl(uint4* ctl, int BS, int t, const CCtl& c) {
    const uint4* s = reinterpret_cast<const uint4*>(&c);
#pragma unroll
    for (int k = 0; k < 4; ++k) ctl[(size_t)k * BS + t] = s[k];
}
// byte j of a 16-byte list held in four registers, without dynamic register indexing
__device__ __forceinline__ int list_byte(const uint32_t w[4], int j) {
    uint32_t v = w[0];
    v = (j >> 2) == 1 ? w[1] : v;
    v = (j >> 2) == 2 ? w[2] : v;
    v = (j >> 2) == 3 ? w[3] : v;
    return (int)((v >> (8 * (j & 3))) & 0xFFu);
}
__device__ __forceinline__ void set_list_byte(uint32_t w[4], int j, int val) {
    const uint32_t m = 0xFFu << (8 * (j & 3)), b = (uint32_t)val << (8 * (j & 3));
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if ((j >> 2) == i) w[i] = (w[i] & ~m) | b;
}

// stream 1: noise of the j-th widening insert of `tree`: component uniform + K standard normals
__device__ __forceinline__ void pw_noise(const TreeParams& p, int64_t tree, int j, float& u, float* z) {
    const uint64_t seed = __ldg(p.seedp);
    u = u32_to_unit(rng_block(seed, tree, 1, j, 0).x);
    for (int b = 0; 2 * b < p.K; ++b) {
        const u32x4 c = rng_block(seed, tree, 1, j, 1 + b);
        const double u1 = ((double)c.x + 0.5) * 2.3283064365386963e-10;
        const double u2 = ((double)c.y + 0.5) * 2.3283064365386963e-10;
        const double rad = sqrt(-2.0 * det::log_(u1));
        double sn, cs;
        det::sincos_(6.283185307179586 * u2, sn, cs);
        z[2 * b] = (float)(rad * cs);
        if (2 * b + 1 < p.K) z[2 * b + 1] = (float)(rad * sn);
    }
}

// MixtureSameFamily.sample with injected noise: component by inverse CDF, x = z*sigma + mu, a = bound*tanh(x)
__device__ __forceinline__ float sample_action(const TreeParams& p, const float* head, float u, const float* z) {
    const int K = p.K;
    int k = 0;
    if (K > 1) {
        float cum = head[2 * K];
        while (k < K - 1 && !(u < cum)) {
            ++k;
            cum = __fadd_rn(cum, head[2 * K + k]);
        }
    }
    const float x = __fadd_rn(__fmul_rn(z[k], head[K + k]), head[k]);
    return p.action_bound > 0.0f ? __fmul_rn(p.action_bound, det::tanhf_(x)) : x;
}

// The same for a compile-time K: the head values stay in registers (the run-time-K version indexes two local arrays dynamically,
// i.e. through local memory, and next to 215 KB of shared memory the whole-search kernel has almost no L1 to catch that: measured
// 5 us of a 22 us tree phase), and only the normal of the SELECTED component is generated (same value as z[k] above).
template <int K>
__device__ __forceinline__ float new_action_k(const TreeParams& p, const float* hptr, int64_t tree, int j) {
    constexpr int HS = (3 * K + 3) / 4 * 4;
    float h[HS];
#pragma unroll
    for (int i = 0; i < HS / 4; ++i) {
        const float4 v = reinterpret_cast<const float4*>(hptr)[i];
        h[4 * i] = v.x; h[4 * i + 1] = v.y; h[4 * i + 2] = v.z; h[4 * i + 3] = v.w;
    }
    const uint64_t seed = __ldg(p.seedp);
    const float u = u32_to_unit(rng_block(seed, tree, 1, j, 0).x);
    int k = 0;
    if (K > 1) {
        float cum = h[2 * K];
#pragma unroll
        for (int i = 1; i < K; ++i)
            if (k == i - 1 && !(u < cum)) {
                k = i;
                cum = __fadd_rn(cum, h[2 * K + i]);
            }
    }
    float mu = h[0], sg = h[K];
#pragma unroll
    for (int i = 1; i < K; ++i)
        if (i == k) { mu = h[i]; sg = h[K + i]; }
    const u32x4 c = rng_block(seed, tree, 1, j, 1 + (k >> 1));
    const double u1 = ((double)c.x + 0.5) * 2.3283064365386963e-10;
    const double u2 = ((double)c.y + 0.5) * 2.3283064365386963e-10;
    const double rad = sqrt(-2.0 * det::log_(u1));
    double sn, cs;
    det::sincos_(6.283185307179586 * u2, sn, cs);
    const float z = (k & 1) ? (float)(rad * sn) : (float)(rad * cs);
    const float x = __fadd_rn(__fmul_rn(z, sg), mu);
    return p.action_bound > 0.0f ? __fmul_rn(p.action_bound, det::tanhf_(x)) : x;
}

// AZG_FLAG_RNG_MT19937: the un-wrapped torch sampling (common.cuh tmt_*; same operation sequence as the oracle's torch_sample_action)
__device__ __forceinline__ double tmt_normal_dev(uint32_t* mt, int& mti) {
    if (mt[MT_N + 3]) {
        mt[MT_N + 3] = 0;
        return __hiloint2double((int)mt[MT_N + 2], (int)mt[MT_N + 1]);
    }
    const double u1 = tmt_uniform_dev(mt, mti), u2 = tmt_uniform_dev(mt, mti);
    const double r = sqrt(2.0 * -det::log_(1.0 - u2));
    double sn, cs;
    det::sincos_(6.283185307179586 * u1, sn, cs);
    const double cached = r * sn;
    mt[MT_N + 1] = (uint32_t)__double2loint(cached);
    mt[MT_N + 2] = (uint32_t)__double2hiint(cached);
    mt[MT_N + 3] = 1;
    return r * cs;
}
__device__ __forceinline__ float new_action_torch(const TreeParams& p, int t, int node) {
    const float* head = p.chead + ((size_t)t * p.R + node) * p.HS;
    uint32_t* mt = p.tmt + (size_t)t * TMT_WORDS;
    int mti = (int)mt[MT_N];
    const int K = p.K;
    int k = 0;
    if (K > 1) {
        float best = 0.0f;
        for (int i = 0; i < K; ++i) {
            const float q = (float)(-det::log_(1.0 - tmt_uniform_dev(mt, mti)));
            const float w = __fdiv_rn(head[2 * K + i], q);
            if (i == 0 || w > best) { best = w; k = i; }
        }
    }
    float z = 0.0f;
    for (int i = 0; i < K; ++i) {
        const float zi = (float)tmt_normal_dev(mt, mti);
        if (i == k) z = zi;
    }
    mt[MT_N] = (uint32_t)mti;
    const float x = __fadd_rn(__fmul_rn(z, head[K + k]), head[k]);
    return p.action_bound > 0.0f ? __fmul_rn(p.action_bound, det::tanhf_(x)) : x;
}

template <bool MT = false>
__device__ __forceinline__ float new_action(const TreeParams& p, int t, int node, int row, int j) {
    if (p.use_tape) return p.tapeA[(size_t)t * p.R + row];
    if (MT) return new_action_torch(p, t, node);
    {
        const float* hptr = p.chead + ((size_t)t * p.R + node) * p.HS;
        const int64_t tree = tree_base(p) + t;
        switch (p.K) {
            case 1: return new_action_k<1>(p, hptr, tree, j);
            case 2: return new_action_k<2>(p, hptr, tree, j);
            case 3: return new_action_k<3>(p, hptr, tree, j);
            case 4: return new_action_k<4>(p, hptr, tree, j);
            default: break;
        }
    }
    // the node's cached policy head (mu[K], sigma[K], prob[K]; HS = 3K rounded up to 4 floats) in 16-byte loads issued before the noise
    float head[3 * AZG_MAX_K];
    const float4* hp = reinterpret_cast<const float4*>(p.chead + ((size_t)t * p.R + node) * p.HS);
#pragma unroll
    for (int i = 0; i < 3 * AZG_MAX_K / 4; ++i)
        if (4 * i < p.HS) {
            const float4 v = hp[i];
            head[4 * i] = v.x; head[4 * i + 1] = v.y; head[4 * i + 2] = v.z; head[4 * i + 3] = v.w;
        }
    float u, z[AZG_MAX_K];
    pw_noise(p, tree_base(p) + t, j, u, z);
    return sample_action(p, head, u, z);
}

__device__ __forceinline__ CHot fresh_hot(double r, float V, float action, uint32_t nn_flags) {
    CHot h;
    h.W = 0.0; h.r = r; h.V = V; h.action = action; h.n_e = 0; h.nn_flags = nn_flags;
    return h;
}

// MCTSContinuous.initialize_search (mcts.py:589-600): new root row, network input = obs(root).  ENV: env.cuh Pendulum |
// MountainCarContinuous (the root is never terminal, even at the goal)
template <class ENV>
__device__ __forceinline__ void c_init(const TreeParams& p, int t) {
    const double th = p.root_state[(size_t)t * 2], thdot = p.root_state[(size_t)t * 2 + 1];
    CRow* root = p.crows + (size_t)t * p.R;
    store_hot(root, fresh_hot(0.0, p.use_tape ? p.tapeV[(size_t)t * p.R] : 0.0f, 0.0f, CROW_EXPANDED));
    store_sec1_new(root, th, thdot);
    p.X[t] = ENV::obs(th, thdot);
    CCtl c;
    memset(&c, 0, sizeof c);
    c.n_rows = 1;
    c.leaf = 0 | LEAF_EVAL;
    store_ctl(p.ctl, p.BS, t, c);
    for (int k = 0; k < 4; ++k) p.ctr[(size_t)k * p.B + t] = 0;
    if (p.rng_mt) {  // random.seed(seed + tree); torch.manual_seed(seed + tree)
        const uint64_t s = __ldg(p.seedp) + (uint64_t)(tree_base(p) + t);
        mt_seed_dev(p.mt + (size_t)t * (MT_N + 1), s);
        tmt_seed_dev(p.tmt + (size_t)t * TMT_WORDS, s);
    }
}
template <class ENV>
__global__ void k_init_continuous(const TreeParams p) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < p.B) c_init<ENV>(p, t);
}

// the add_pw_action(root) that precedes the rollout loop (mcts.py:673); runs after the root evaluation
template <bool MT = false>
__device__ __forceinline__ void c_root_insert(const TreeParams& p, int t) {
    CRow* rows = p.crows + (size_t)t * p.R;
    CCtl c = load_ctl(p.ctl, p.BS, t);
    const float a = new_action<MT>(p, t, 0, 1, 0);
    store_hot(p.et + t, fresh_hot(0.0, 0.0f, a, 0));  // root child 0
    store_sec1_new(rows + 1, 0.0, 0.0);
    c.root_kids[0] = 1;
    c.root_nk = 1;
    c.n_rows = 2;
    c.pw = 1;
    c.root_V = rows[0].V;  // written by the root evaluation
    c.root_nn = 0;
    store_ctl(p.ctl, p.BS, t, c);
}
__global__ void k_root_insert_continuous(const TreeParams p) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p.B) return;
    if (p.rng_mt) c_root_insert<true>(p, t);
    else c_root_insert<false>(p, t);
}

#define KIND_INSERT 0    // progressive widening: create a new edge below `cur`, then its node
#define KIND_EXPAND 1    // an existing edge without a node (only the root's first edge when c_pw > 1)
#define KIND_TERMINAL 2  // the trace ended on an existing terminal node
#define KIND_ERROR 3

// UCT over the nk <= 16 children of a node; returns the selected index (mcts.py:729-741 + helpers.argmax + epsilon_greedy).
// Child j's hot sector is et[j] for the root and rows[kids[j]] otherwise.  Only the two fields the score needs (W, n) are
// gathered, four children per round trip; the score loop is ROLLED (the four gathered pairs rotate through one set of
// registers) and there is one instance of it for root and inner nodes: the first version unrolled 16 children x 2 call sites
// x two inlined IEEE divisions into 5000 SASS instructions, which the whole-search kernel (qmlp2.cuh) paid for in instruction
// fetch on the evaluation warps.
__device__ __forceinline__ const CHot* child_hot(const CHot* et, int BS, const CRow* rows, const uint32_t kw[4], bool is_root, int j) {
    return is_root ? et + (size_t)j * BS : reinterpret_cast<const CHot*>(rows + list_byte(kw, j));  // et = &table[0][t]
}
__device__ __forceinline__ int uct_select(const TreeParams& p, const Tabs& tb, int64_t tree, int nk, uint32_t cur_nn, float cur_V, int& draws,
                                          bool& nan, const CHot* et, const CRow* rows, const uint32_t kw[4], bool is_root, uint32_t* mt = nullptr) {
    const double sq = sqrt_small((int)cur_nn + 1, tb.sq, tb.n);
    double best = -CUDART_INF;
    uint32_t win = 0;
#pragma unroll 1
    for (int w0 = 0; w0 < nk; w0 += 4) {
        double W[4];
        int n[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const uint4 q = *reinterpret_cast<const uint4*>(child_hot(et, p.BS, rows, kw, is_root, w0 + i < nk ? w0 + i : w0));
            W[i] = __hiloint2double((int)q.y, (int)q.x);  // CHot::W
            n[i] = (int)q.z;                              // CHot::n_e
        }
        const int m = min(4, nk - w0);
#pragma unroll 1
        for (int i = 0; i < m; ++i) {
            const double Q = n[0] > 0 ? div_small(W[0], n[0], tb.rcp, tb.n) : (double)cur_V;
            const double u = Q + p.c_uct * div_small(sq, n[0] + 1, tb.rcp, tb.n);  // mcts.py:731-732
            nan |= (u != u);
            if (u > best) { best = u; win = 1u << (w0 + i); }
            else if (u == best) win |= 1u << (w0 + i);
            W[0] = W[1]; W[1] = W[2]; W[2] = W[3];
            n[0] = n[1]; n[1] = n[2]; n[2] = n[3];
        }
    }
    bool random_pick = false;
    if (mt) {  // AZG_FLAG_RNG_MT19937: CPython's generator (random(): two outputs; choice / randint: _randbelow_with_getrandbits)
        int mti = (int)mt[MT_N];
        if (p.epsilon != 0) random_pick = mt_random_dev(mt, mti, draws) < p.epsilon;
        const int nwm = random_pick ? nk : __popc(win);
        const int pk = nwm > 0 ? mt_below_dev(mt, mti, draws, nwm) : 0;
        mt[MT_N] = (uint32_t)mti;
        if (random_pick) return pk;
        return nwm > 0 ? (int)__fns(win, 0, pk + 1) : 0;
    }
    if (p.epsilon != 0) {  // epsilon_greedy (mcts.py:175-195)
        const double x = (double)u32_to_unit(rng_select_u32(p, tree, draws++));
        random_pick = x < p.epsilon;
    }
    // random.choice(winners) / random.randint: the draw is consumed even when there is a single winner
    const int nw = random_pick ? nk : __popc(win);
    const int pick = nw > 1 ? u32_to_index(rng_select_u32(p, tree, draws), nw) : 0;
    ++draws;
    if (random_pick) return pick;
    if (nw == 1) return __ffs((int)win) - 1;  // the usual case without the software find-nth-set routine
    return nw > 0 ? (int)__fns(win, 0, pick + 1) : 0;
}

// one simulation step of tree t: backup of the previous simulation (BACKUP), then descent + expansion of the next (SELECT).
// Shared by k_step_continuous (one launch per simulation) and the whole-search kernel k_search_fused (fused.cuh).
// MT: AZG_FLAG_RNG_MT19937 (CPython's and torch's generators, 5 KB of state per tree in HBM: a compatibility mode that the one-launch-
// per-simulation kernel alone instantiates; the whole-search kernels are built without it)
template <class ENV, bool MT = false>
__device__ __forceinline__ void c_step(const TreeParams& p, const Tabs& tb, int t, const bool BACKUP, const bool SELECT) {
    CRow* rows = p.crows + (size_t)t * p.R;
    CHot* et = p.et + t;  // root child j: et[j * BS]
    uint8_t* path_ovf = p.path + (size_t)t * p.R;
    // per-tree counters: read here, written at the end (a read-modify-write at the end exposed the load latency)
    uint32_t ctr_levels = 0, ctr_scanned = 0;
    if (SELECT) { ctr_levels = p.ctr[t]; ctr_scanned = p.ctr[(size_t)p.B + t]; }
    TP_BEGIN();
    CCtl c = load_ctl(p.ctl, p.BS, t);
    uint32_t pathw[4];
    memcpy(pathw, c.path, 16);
    TP_STAMP(0);
    if (BACKUP) {
        // backprop (mcts.py:241-267) along the recorded path.  leafR already holds r_leaf + gamma*V_leaf
        // (the f32 product of NEP 50, added by the evaluation kernel's epilogue).
        const int d = c.depth;
        double Rv = c.leafR;
        for (int i = d - 1; i >= 0; --i) {
            void* hp = i == 0 ? (void*)(et + (size_t)c.j0 * p.BS) : (void*)(rows + (i < 16 ? list_byte(pathw, i) : (int)path_ovf[i]));
            const CHot h = load_hot(hp);
            if (i != d - 1) Rv = h.r + p.gamma * Rv;
            const double Wn = h.W + Rv;  // Action.update (states.py:97-112): W, n and the child node's n in one 16-byte store
            *reinterpret_cast<uint4*>(hp) = make_uint4((uint32_t)__double2loint(Wn), (uint32_t)__double2hiint(Wn), (uint32_t)(h.n_e + 1),
                                                       h.nn_flags + (i < d - 1 ? 1u : 0u));
        }
        if (d > 0) c.root_nn += 1;  // root.n
    }
    TP_STAMP(1);

    if (SELECT) {
        const int64_t tree = tree_base(p) + t;
        int draws = c.draws, n_rows = c.n_rows, pwc = c.pw;
        int cur = 0, sel = -1, kind = KIND_ERROR, depth = 0, nk = c.root_nk;
        uint32_t cur_nn = (uint32_t)c.root_nn;
        float cur_V = c.root_V, sel_action = 0.0f;
        double leaf_r = 0.0, cur_th = 0.0, cur_thdot = 0.0;
        uint32_t kw[4], rootk[4];
        memcpy(rootk, c.root_kids, 16);
        kw[0] = rootk[0]; kw[1] = rootk[1]; kw[2] = rootk[2]; kw[3] = rootk[3];
        uint32_t levels = 0, scanned = 0;
        bool nan = false;
        int jsel = 0;
        while (true) {
            ++levels;
            if (tb.pw[cur_nn] - nk > 0) { kind = KIND_INSERT; break; }  // states.py:252-275
            jsel = uct_select(p, tb, tree, nk, cur_nn, cur_V, draws, nan, et, rows, kw, cur == 0, MT ? p.mt + (size_t)t * (MT_N + 1) : nullptr);
            sel = list_byte(kw, jsel);
            const CHot sh = load_hot(child_hot(et, p.BS, rows, kw, cur == 0, jsel));  // the line was gathered a moment ago
            // requested together with sh (one round trip instead of two); used only if the descent enters the node
            const CSec1 s1 = load_sec1(rows + sel);
            scanned += nk;
            if (depth == 0) c.j0 = (uint8_t)jsel;
            if (depth < 16) set_list_byte(pathw, depth, sel); else path_ovf[depth] = (uint8_t)sel;
            ++depth;
            if (!(sh.nn_flags & CROW_EXPANDED)) { kind = KIND_EXPAND; sel_action = sh.action; break; }
            const bool from_root = cur == 0;
            cur = sel;
            cur_nn = sh.nn_flags & CROW_NMASK;
            cur_V = sh.V;
            if (sh.nn_flags & CROW_TERMINAL) { kind = KIND_TERMINAL; leaf_r = sh.r; (void)from_root; break; }
            kw[0] = s1.kw[0]; kw[1] = s1.kw[1]; kw[2] = s1.kw[2]; kw[3] = s1.kw[3];
            nk = (int)(kw[3] >> 24);
            cur_th = s1.th; cur_thdot = s1.thdot;
        }
        TP_STAMP(2);
        if (nan) { atomicOr(p.err, ERR_NAN); kind = KIND_ERROR; }
        if (kind == KIND_INSERT && (n_rows >= p.R || n_rows >= 255 || nk >= (cur == 0 ? CROOT_MAX_KIDS : CROW_MAX_KIDS))) {
            atomicOr(p.err, ERR_CAPACITY);
            kind = KIND_ERROR;
        }

        // ---- expansion: all lanes are reconverged here, so the f64 work below runs on full warps ----
        const bool parent_is_root = cur == 0;  // (for KIND_EXPAND / KIND_INSERT `cur` is the parent of `sel`)
        if (kind == KIND_INSERT) {
            // add_pw_action (mcts.py:625-654): the new edge is selected immediately (mcts.py:725-727)
            sel = n_rows++;
            sel_action = new_action<MT>(p, t, cur, sel, pwc++);
            jsel = nk;
            if (parent_is_root) {
                set_list_byte(rootk, nk, sel);
                c.root_nk = (uint8_t)(nk + 1);
            } else {
                set_list_byte(kw, nk, sel);  // the node's child list + count (top byte) go back in one 16-byte store
                kw[3] = (kw[3] & 0x00FFFFFFu) | ((uint32_t)(nk + 1) << 24);
                reinterpret_cast<uint4*>(rows + cur)[2] = make_uint4(kw[0], kw[1], kw[2], kw[3]);
            }
            if (depth == 0) c.j0 = (uint8_t)jsel;
            if (depth < 16) set_list_byte(pathw, depth, sel); else path_ovf[depth] = (uint8_t)sel;
            ++depth;
        }
        TP_STAMP(3);
        if (kind == KIND_INSERT || kind == KIND_EXPAND) {
            if (parent_is_root) {  // the root's state sits in row 0 (read only when the tree grows at the root)
                const CSec1 s0 = load_sec1(rows);
                cur_th = s0.th; cur_thdot = s0.thdot;
            }
            double nth, nthdot, rew;
            const bool term = ENV::step(cur_th, cur_thdot, sel_action, nth, nthdot, rew);
            const double r = rew / AZG_PENDULUM_R_SCALE;  // mcts.py:687: Pendulum's scale, whatever the env
            const uint32_t fl = CROW_EXPANDED | (term ? CROW_TERMINAL : 0u);
            float V = 0.0f;
            if (p.use_tape && !term) V = p.tapeV[(size_t)t * p.R + sel];
            void* hp = parent_is_root ? (void*)(et + (size_t)jsel * p.BS) : (void*)(rows + sel);
            if (kind == KIND_INSERT) {
                store_hot(hp, fresh_hot(r, V, sel_action, fl));
            } else {
                CHot* h = reinterpret_cast<CHot*>(hp);
                h->r = r; h->V = V; h->nn_flags = fl;
            }
            store_sec1_new(rows + sel, nth, nthdot);
            p.X[t] = ENV::obs(nth, nthdot);
            c.leaf = sel | LEAF_EVAL | (term ? LEAF_TERMINAL : 0) | (parent_is_root ? (LEAF_ROOTCHILD | (jsel << LEAF_J_SHIFT)) : 0);
            // first backup step R = r + gamma*V: with tapes V is known here, otherwise the evaluation kernel adds it
            c.leafR = p.use_tape ? r + (double)__fmul_rn(p.gamma_f32, V) : r;
        } else if (kind == KIND_TERMINAL) {
            c.leaf = cur;
            c.leafR = leaf_r + (double)__fmul_rn(p.gamma_f32, 0.0f);
            p.ctr[(size_t)2 * p.B + t] += 1;
        } else {
            c.leaf = 0;
            depth = 0;
        }
        c.n_rows = (uint8_t)n_rows;
        c.draws = draws;
        c.pw = (uint16_t)pwc;
        c.depth = (uint8_t)depth;
        p.ctr[t] = ctr_levels + levels;
        p.ctr[(size_t)p.B + t] = ctr_scanned + scanned;
        memcpy(c.root_kids, rootk, 16);
    }
    memcpy(c.path, pathw, 16);
    store_ctl(p.ctl, p.BS, t, c);
    TP_STAMP(4);
}
template <class ENV, bool BACKUP, bool SELECT>
__global__ void __launch_bounds__(128) k_step_continuous(const TreeParams p) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const Tabs tb = {p.pw_table, p.rcp_tab, p.sqrt_tab, AZG_TAB};
    if (t >= p.B) return;
    if (p.rng_mt) c_step<ENV, true>(p, tb, t, BACKUP, SELECT);
    else c_step<ENV, false>(p, tb, t, BACKUP, SELECT);
}

// numpy pairwise summation for n <= 128 (np.sum in get_on_policy_value_target, mcts.py:111)
__device__ __forceinline__ double np_sum(const double* a, int n) {
    if (n < 8) {
        double r = 0.;
        for (int i = 0; i < n; ++i) r += a[i];
        return r;
    }
    double r[8];
    for (int k = 0; k < 8; ++k) r[k] = a[k];
    int i;
    for (i = 8; i < n - (n % 8); i += 8)
        for (int k = 0; k < 8; ++k) r[k] += a[i + k];
    double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; ++i) res += a[i];
    return res;
}

// MCTS.return_results (mcts.py:269-307): root children in insertion order = the root edge table, one thread per tree
__global__ void k_results_continuous(const TreeParams p, int cmax, float* actions, int32_t* counts, double* Q, double* Vt,
                                     int32_t* nchild) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p.B) return;
    const CHot* et = p.et + t;
    const CCtl c = load_ctl(p.ctl, p.BS, t);
    const float Vroot = c.root_V;
    const int nk = min((int)c.root_nk, cmax);
    double q[CROOT_MAX_KIDS];
    int32_t cn[CROOT_MAX_KIDS];
    for (int j = 0; j < nk; ++j) {
        const CHot h = load_hot(et + (size_t)j * p.BS);
        q[j] = h.n_e > 0 ? h.W / (double)h.n_e : (double)Vroot;
        cn[j] = h.n_e;
        actions[(size_t)t * cmax + j] = h.action;
        counts[(size_t)t * cmax + j] = h.n_e;
        Q[(size_t)t * cmax + j] = q[j];
    }
    for (int j = nk; j < cmax; ++j) {
        actions[(size_t)t * cmax + j] = 0.0f;
        counts[(size_t)t * cmax + j] = 0;
        Q[(size_t)t * cmax + j] = 0.0;
    }
    nchild[t] = nk;
    double v = 0.0;
    if (nk > 0) {
        if (p.v_target == 1) {
            long long tot = 0;
            for (int j = 0; j < nk; ++j) tot += cn[j];
            for (int j = 0; j < nk; ++j) q[j] = ((double)cn[j] / (double)tot) * q[j];
            v = np_sum(q, nk);
        } else {
            v = q[0];
            for (int j = 1; j < nk; ++j) v = q[j] > v ? q[j] : v;
        }
    }
    Vt[t] = v;
}

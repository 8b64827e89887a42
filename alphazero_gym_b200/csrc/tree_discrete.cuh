// tree_discrete.cuh -- backup + PUCT select + expansion for the discrete (CartPole) tree.
//
// Reference: MCTSDiscrete.search (mcts.py:418-462), selectionUCT (:464-493), epsilon_greedy (:175-195),
// helpers.argmax (helpers.py:30-52), MCTS.backprop (mcts.py:241-267), Action.update (states.py:97-112),
// expansion (mcts.py:215-238).
//
// Mapping: fan-out is A = 2, so a warp-wide argmax would idle 30 lanes; instead one THREAD owns one tree
// and a warp advances 32 trees in lockstep.  A node visit is one 64 B row = two full 32 B sectors, read
// with 4 x LDG.128; the level loop is a chain of dependent row loads (parent -> chosen child).  The env
// step runs after the loop so that all 32 lanes execute the f64 dynamics together.
#pragma once
#include "common.cuh"
#include "env.cuh"

__device__ __forceinline__ DRow load_drow(const DRow* p) {
    DRow r;
    const uint4* s = reinterpret_cast<const uint4*>(p);
    uint4* d = reinterpret_cast<uint4*>(&r);
    d[0] = s[0]; d[1] = s[1]; d[2] = s[2]; d[3] = s[3];
    return r;
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
// line 0 of a three-action row: everything the descent reads
__device__ __forceinline__ void load_line0(D3Row* r, const D3Row* p) {
    const uint4* s = reinterpret_cast<const uint4*>(p);
    uint4* d = reinterpret_cast<uint4*>(r);
    d[0] = s[0]; d[1] = s[1]; d[2] = s[2]; d[3] = s[3];
}

// a fresh three-action row: no edges visited, no children
__device__ __forceinline__ D3Row d3_row(uint16_t parent, int paction, double r, bool term) {
    D3Row nr;
    memset(&nr, 0, sizeof nr);
    nr.child[0] = nr.child[1] = nr.child[2] = DROW_NONE;
    nr.flags = term ? ROW_TERMINAL : 0;
    nr.r = r;
    nr.parent = parent;
    nr.paction = (uint8_t)paction;
    return nr;
}

// root row + first network input (MCTSDiscrete.initialize_search, mcts.py:364-383)
template <class ENV>
__device__ __forceinline__ void d_init(const TreeParams& p, int t) {
    const double* s = p.root_state + (size_t)t * ENV::HS;  // the root's hidden state
    double* st = p.dstate + (size_t)t * p.R * 4;
    if constexpr (ENV::A == 2) {
        DRow row;
        row.W[0] = row.W[1] = 0.0;
        row.r = 0.0;
        row.n_e[0] = row.n_e[1] = 0;
        row.prior[0] = row.prior[1] = 0.0f;
        row.V = 0.0f;
        row.node_n = p.root_n_init ? p.root_n_init[t] : 0;
        row.child[0] = row.child[1] = DROW_NONE;
        row.parent = DROW_NONE;
        row.paction = 0;
        row.flags = 0;
        row.pad[0] = row.pad[1] = 0;
        if (p.use_tape) {
            row.V = p.tapeV[(size_t)t * p.R];
            row.prior[0] = p.tapeP[(size_t)t * p.R * 2];
            row.prior[1] = p.tapeP[(size_t)t * p.R * 2 + 1];
        }
        p.drows[(size_t)t * p.R] = row;
        st[0] = s[0]; st[1] = s[1]; st[2] = s[2]; st[3] = s[3];
        p.X[t] = make_float4((float)s[0], (float)s[1], (float)s[2], (float)s[3]);
    } else {
        D3Row row = d3_row(DROW_NONE, 0, 0.0, false);
        row.node_n = p.root_n_init ? p.root_n_init[t] : 0;
        if (p.use_tape) {
            row.V = p.tapeV[(size_t)t * p.R];
            for (int k = 0; k < 3; ++k) row.prior[k] = p.tapeP[(size_t)t * p.R * 3 + k];
        }
        reinterpret_cast<D3Row*>(p.drows)[(size_t)t * p.R] = row;
#pragma unroll
        for (int k = 0; k < ENV::HS; ++k) st[k] = s[k];
        ENV::input(s, p.X + (size_t)t * ENV::XW);  // the root's observation, from its hidden state
    }
    p.leaf[t] = 0 | LEAF_EVAL;
    p.n_rows[t] = 1;
    p.draws[t] = 0;
    if (p.rng_mt) mt_seed_dev(p.mt + (size_t)t * (MT_N + 1), __ldg(p.seedp) + (uint64_t)(tree_base(p) + t));  // random.seed(seed + tree)
    for (int k = 0; k < 4; ++k) p.ctr[(size_t)k * p.B + t] = 0;
}
template <class ENV>
__global__ void k_init_discrete(const TreeParams p) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < p.B) d_init<ENV>(p, t);
}

// one simulation step of tree t: backup of the previous simulation (BACKUP), then descent + expansion of the next (SELECT).
// Shared by k_step_discrete (one launch per simulation) and the whole-search kernels (qmlp2.cuh, search_wg.cuh).
// ENV::A = 2 (CartPole): DRow, path entries (row << 1 | action).  ENV::A = 3 (MountainCar, Acrobot): D3Row, path entries
// (row << 2 | action); the descent reads line 0 of a row, the backup also reads r from line 1.
template <class ENV>
__device__ __forceinline__ void d_step(const TreeParams& p, const Tabs& tb, int t, const bool BACKUP, const bool SELECT) {
    constexpr int A = ENV::A, PSH = A == 2 ? 1 : 2;  // path entry: row << PSH | action
    DRow* rows = p.drows + (size_t)t * p.R;
    D3Row* rows3 = reinterpret_cast<D3Row*>(p.drows) + (size_t)t * p.R;

    uint16_t* path = p.dpath + (size_t)t * p.R;
    TP_BEGIN();
    if (BACKUP) {
        // R = leaf.V; up the path: R = node.r + gamma*R; edge.n += 1; edge.W += R; parent.n += 1 (mcts.py:241-267).
        // The select step recorded the path (row, action) root -> leaf, so the row addresses are known up front and the rows are
        // fetched four at a time; following the parent links instead made every level a dependent L2 round trip, and CartPole
        // traces are 8 levels deep on average (tens in the deepest tree of a warp).
        const int leaf = p.leaf[t] & LEAF_ROW_MASK;
        const int d = p.ddepth[t];
        double Rv, r;
        if constexpr (A == 2) {
            const DRow lr = load_drow(rows + leaf);
            Rv = (double)lr.V;
            r = lr.r;
        } else {
            Rv = (double)rows3[leaf].V;
            r = rows3[leaf].r;
        }
#pragma unroll 1
        for (int base = d - 1; base >= 0; base -= 4) {
            if constexpr (A == 2) {
                DRow q[4];
                int pe[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    pe[k] = base - k >= 0 ? (int)path[base - k] : 0;
                    q[k] = load_drow(rows + (pe[k] >> 1));
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (base - k >= 0) {
                        DRow* pr = rows + (pe[k] >> 1);
                        const int pa = pe[k] & 1;
                        Rv = r + p.gamma * Rv;
                        pr->W[pa] = (pa ? q[k].W[1] : q[k].W[0]) + Rv;
                        pr->n_e[pa] = (pa ? q[k].n_e[1] : q[k].n_e[0]) + 1;
                        pr->node_n = q[k].node_n + 1;
                        r = q[k].r;
                    }
                }
            } else {  // only the four words the backup touches per level: the edge's W and n, node.n (line 0) and r (line 1)
                double qW[4], qr[4];
                int qn[4], qnn[4], pe[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    pe[k] = base - k >= 0 ? (int)path[base - k] : 0;
                    const D3Row* q = rows3 + (pe[k] >> 2);
                    const int pa = pe[k] & 3;
                    qW[k] = q->W[pa];
                    qn[k] = q->n_e[pa];
                    qnn[k] = q->node_n;
                    qr[k] = q->r;
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (base - k >= 0) {
                        D3Row* pr = rows3 + (pe[k] >> 2);
                        const int pa = pe[k] & 3;
                        Rv = r + p.gamma * Rv;
                        pr->W[pa] = qW[k] + Rv;
                        pr->n_e[pa] = qn[k] + 1;
                        pr->node_n = qnn[k] + 1;
                        r = qr[k];
                    }
                }
            }
        }
    }

    TP_STAMP(1);
    if (SELECT) {
        const int64_t tree = tree_base(p) + t;
        int draws = p.draws[t];
        int cur = 0;
        // the node being descended: a DRow, or line 0 of a D3Row
        DRow row;
        D3Row row3;
        if constexpr (A == 2) row = load_drow(rows);
        else load_line0(&row3, rows3);
        int a = -1;
        uint32_t levels = 0;
        uint32_t xr[4] = {0, 0, 0, 0};
        uint32_t* mt = p.rng_mt ? p.mt + (size_t)t * (MT_N + 1) : nullptr;
        int mti = p.rng_mt ? (int)mt[MT_N] : 0;
        bool nan = false;
        while (true) {
            // CartPole: both children are LOADED while the scores are computed (32 registers): the level costs max(round trip,
            // arithmetic) instead of their sum, and the next level's children are requested the moment the choice is made.
            // MountainCar: holding line 0 of three children (48 registers) spilled in the warpgroup kernel (search_wg.cuh), so the
            // three lines are prefetched into L2 instead and only the chosen one is loaded
            uint4 k0[4], k1[4];
            int c0, c1, c2 = DROW_NONE;
            if constexpr (A == 2) {
                c0 = row.child[0], c1 = row.child[1];
                const uint4* s0 = reinterpret_cast<const uint4*>(rows + (c0 != DROW_NONE ? c0 : cur));
                const uint4* s1 = reinterpret_cast<const uint4*>(rows + (c1 != DROW_NONE ? c1 : cur));
#pragma unroll
                for (int q = 0; q < 4; ++q) { k0[q] = s0[q]; k1[q] = s1[q]; }
            } else {
                c0 = row3.child[0], c1 = row3.child[1], c2 = row3.child[2];
                if (c0 != DROW_NONE) prefetch_l2(rows3 + c0);
                if (c1 != DROW_NONE) prefetch_l2(rows3 + c1);
                if (c2 != DROW_NONE) prefetch_l2(rows3 + c2);
            }
            // UCT_a = Q_a + prior_a*c_uct*(sqrt(node.n+1)/(n_a+1))   (mcts.py:483-484)
            const double sq = sqrt_small((A == 2 ? row.node_n : row3.node_n) + 1, tb.sq, tb.n);
            double u[A];
#pragma unroll
            for (int i = 0; i < A; ++i) {
                const int n = A == 2 ? row.n_e[i] : row3.n_e[i];
                const double Q = n > 0 ? div_small(A == 2 ? row.W[i] : row3.W[i], n, tb.rcp, tb.n) : (double)(A == 2 ? row.V : row3.V);
                const float pr = A == 2 ? row.prior[i] : row3.prior[i];
                const double pc = p.puct_f32 ? (double)__fmul_rn(pr, (float)p.c_uct) : (double)pr * p.c_uct;
                u[i] = Q + pc * div_small(sq, n + 1, tb.rcp, tb.n);
            }
            if constexpr (A == 2) nan |= (u[0] != u[0]) || (u[1] != u[1]);
            else nan |= (u[0] != u[0]) || (u[1] != u[1]) || (u[2] != u[2]);
#ifdef AZG_TREE_PROF
            if (u[0] + u[1] == 12345.678) atomicOr(p.err, 0);  // (profiling builds: the scores are complete before the stamp)
            TP_STAMP(5);
#endif
            bool random_pick = false;
            if (p.epsilon != 0 && p.rng_mt) {
                random_pick = mt_random_dev(mt, mti, draws) < p.epsilon;
            } else if (p.epsilon != 0) {  // epsilon_greedy: random.random() < eps -> random.randint(0, A-1)
                // every level consumes exactly two draws (random(), then randint or choice), so the random() of the next four
                // levels are draws + 0, 2, 4, 6: generated together (the generator was half of a level's dependent chain)
                const int k = (int)(levels & 3u);
                if (k == 0) rng_select_u32x4(__ldg(p.seedp), tree, draws, 2, xr);
                const uint32_t xk = k == 0 ? xr[0] : (k == 1 ? xr[1] : (k == 2 ? xr[2] : xr[3]));
                ++draws;
                const double x = (double)u32_to_unit(xk);
                random_pick = x < p.epsilon;
            }
            if constexpr (A == 2) {
                if (p.rng_mt) {  // randint(0, 1), or choice over the 1 or 2 winners (which also draws for a single winner)
                    if (random_pick) a = mt_below_dev(mt, mti, draws, 2);
                    else if (u[0] == u[1]) a = mt_below_dev(mt, mti, draws, 2);
                    else { (void)mt_below_dev(mt, mti, draws, 1); a = u[1] > u[0] ? 1 : 0; }
                } else if (random_pick) {
                    a = u32_to_index(rng_select_u32(p, tree, draws++), 2);
                } else {
                    // argmax with random tie-break: one draw is consumed even for a single winner
                    if (u[0] == u[1]) a = u32_to_index(rng_select_u32(p, tree, draws), 2);
                    else a = u[1] > u[0] ? 1 : 0;
                    ++draws;
                }
            } else {
                // helpers.argmax: winners = the indices of max(u) in ascending order; random.choice(winners), one draw even for a
                // single winner (a NaN score leaves no winner: ERR_NAN is raised and the pick is immaterial)
                double m = u[0];
                m = u[1] > m ? u[1] : m;
                m = u[2] > m ? u[2] : m;
                const int w0 = u[0] == m, w1 = u[1] == m, nw = w0 + w1 + (u[2] == m);
                int pick = 0;
                if (p.rng_mt) {  // randint(0, 2) / CPython's _randbelow(n_winners)
                    if (random_pick) a = mt_below_dev(mt, mti, draws, 3);
                    else pick = mt_below_dev(mt, mti, draws, nw > 0 ? nw : 1);
                } else if (random_pick) {
                    a = u32_to_index(rng_select_u32(p, tree, draws++), 3);
                } else {
                    if (nw > 1) pick = u32_to_index(rng_select_u32(p, tree, draws), nw);
                    ++draws;
                }
                if (!random_pick) a = (w0 && pick == 0) ? 0 : ((w1 && pick == w0) ? 1 : 2);
            }
#ifdef AZG_TREE_PROF
            if (a == 77) atomicOr(p.err, 0);
            TP_STAMP(6);
            if ((threadIdx.x & 31) == 0 && p.prof) atomicAdd(p.prof + 7, 1ull);
#endif
            path[levels] = (uint16_t)((cur << PSH) | a);
            ++levels;
            const int child = A == 2 ? (a ? c1 : c0) : (a == 0 ? c0 : (a == 1 ? c1 : c2));
            if (child == DROW_NONE) break;  // expansion
            cur = child;
            if constexpr (A == 2) {
                uint4* d = reinterpret_cast<uint4*>(&row);
#pragma unroll
                for (int q = 0; q < 4; ++q) d[q] = a ? k1[q] : k0[q];
                if (row.flags & ROW_TERMINAL) { a = -1; break; }  // trace ends on an existing terminal node
            } else {
                load_line0(&row3, rows3 + child);
                if (row3.flags & ROW_TERMINAL) { a = -1; break; }
            }
#ifdef AZG_TREE_PROF
            if ((A == 2 ? row.node_n : row3.node_n) == -77) atomicOr(p.err, 0);  // (the next row has arrived)
            TP_STAMP(3);
#endif
        }
        TP_STAMP(2);
        if (nan) atomicOr(p.err, ERR_NAN);
        if (p.rng_mt) mt[MT_N] = (uint32_t)mti;
        p.ddepth[t] = (int)levels;  // edges between the root and the leaf (the new node, or the existing terminal node the trace ended on)
        p.draws[t] = draws;
        p.ctr[t] += levels;
        p.ctr[(size_t)p.B + t] += levels * A;
        if (a >= 0) {
            const int child = p.n_rows[t];
            if (child >= p.R) { atomicOr(p.err, ERR_CAPACITY); p.leaf[t] = cur; return; }
            p.n_rows[t] = child + 1;
            double* st = p.dstate + ((size_t)t * p.R + cur) * 4;
            bool term;
            if constexpr (A == 2) {
                const double s[4] = {st[0], st[1], st[2], st[3]};
                double o[4], rew;
                term = env::cartpole_step(s, a, o, rew);
                rew = term ? p.reward_terminal : p.reward_step;  // rl/wrappers.py (1.0 / 1.0 without wrappers)
                double* so = p.dstate + ((size_t)t * p.R + child) * 4;
                so[0] = o[0]; so[1] = o[1]; so[2] = o[2]; so[3] = o[3];
                DRow nr;
                nr.W[0] = nr.W[1] = 0.0;
                nr.r = rew;
                nr.n_e[0] = nr.n_e[1] = 0;
                nr.prior[0] = nr.prior[1] = 0.0f;
                nr.V = 0.0f;
                nr.node_n = 0;
                nr.child[0] = nr.child[1] = DROW_NONE;
                nr.parent = (uint16_t)cur;
                nr.paction = (uint8_t)a;
                nr.flags = term ? ROW_TERMINAL : 0;
                nr.pad[0] = nr.pad[1] = 0;
                if (p.use_tape) {
                    const size_t ti = (size_t)t * p.R + child;
                    nr.V = term ? 0.0f : p.tapeV[ti];
                    nr.prior[0] = p.tapeP[ti * 2];
                    nr.prior[1] = p.tapeP[ti * 2 + 1];
                }
                rows[child] = nr;
                rows[cur].child[a] = (uint16_t)child;
                p.X[t] = make_float4((float)o[0], (float)o[1], (float)o[2], (float)o[3]);
            } else {
                double h[ENV::HS], o[ENV::HS], rew;
                bool capped = false;
#pragma unroll
                for (int k = 0; k < ENV::HS; ++k) h[k] = st[k];
                term = ENV::expand(h, a, o, rew, capped);  // Node.r = the env's reward
                if (capped) atomicOr(p.err, ERR_WRAP);
                double* so = p.dstate + ((size_t)t * p.R + child) * 4;
#pragma unroll
                for (int k = 0; k < ENV::HS; ++k) so[k] = o[k];
                D3Row nr = d3_row((uint16_t)cur, a, rew, term);
                if (p.use_tape) {
                    const size_t ti = (size_t)t * p.R + child;
                    nr.V = term ? 0.0f : p.tapeV[ti];
                    for (int k = 0; k < 3; ++k) nr.prior[k] = p.tapeP[ti * 3 + k];
                }
                rows3[child] = nr;
                rows3[cur].child[a] = (uint16_t)child;
                ENV::input(o, p.X + (size_t)t * ENV::XW);
            }
            p.leaf[t] = child | LEAF_EVAL | (term ? LEAF_TERMINAL : 0);
        } else {
            p.leaf[t] = cur;
            p.ctr[(size_t)2 * p.B + t] += 1;
        }
        TP_STAMP(4);
    }
}

template <class ENV, bool BACKUP, bool SELECT>
__global__ void __launch_bounds__(128) k_step_discrete(const TreeParams p) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const Tabs tb = {p.pw_table, p.rcp_tab, p.sqrt_tab, AZG_TAB};
    if (t < p.B) d_step<ENV>(p, tb, t, BACKUP, SELECT);
}

// ---- shared-memory-resident trees (whole-search kernel, thin batches: qmlp2.cuh TSM) -----------------------------------------------
// At BASELINE config 3 (4096 CartPole trees x 50 simulations) a B200 holds 28 trees per SM, and their rows -- 28 x 52 x 64 B = 93 KB --
// fit next to the evaluation's operands in the SM's 227 KB of shared memory.  The tree step is a chain of dependent row visits
// (CartPole traces are ~10 levels deep) and with the rows in HBM / L2 every visit is a ~700-cycle round trip executed by a lone
// warp: 25 us of a 32 us simulation (profiles/README.md r2e).  From shared memory a visit is ~30 cycles, the backup can simply follow
// the parent links again (mcts.py:241-267 as written) and needs no recorded path, and the per-tree scalars never leave the SM.
// Same arithmetic in the same order as d_step: results are bit-identical.  The rows are copied to p.drows when the search ends
// (k_results_discrete, azg_dump_tree, the self-play step and tree reuse read them there); the env states stay in p.dstate.
struct __align__(16) STree {  // per-tree scalars (p.leaf / p.n_rows / p.draws / p.ctr / p.ddepth of the global-memory path)
    int32_t n_rows, draws;
    uint32_t levels;        // levels descended, summed over the search
    uint16_t terms, depth;  // simulations that ended on an existing terminal node; length of the current simulation's path
};
struct SmTrees {
    DRow* rows;      // [trees][R]
    STree* st;       // [trees]
    float4* X;       // [trees]  network input of the leaf
    int32_t* leaf;   // [trees]  LEAF_* word
    uint16_t* path;  // [trees][R]  recorded path of the current simulation
    float* part;     // [4][PO_PAD][trees]  head partial sums of the column quarters (qmlp2.cuh q2_heads_tsm): the tree phase finishes the rows
};
// Everything the tree phase needs, written once per launch into shared memory by the kernel and copied into registers when the
// phase starts: with the kernel's own parameter blocks (and ~70 registers of the epilogue live across the phase) the compiler
// rematerialised every address inside the level loop -- 75 instructions per level (profiles/README.md r2i)
struct __align__(16) DsCtx {
    SmTrees sm;
    double* dstate;      // env states of the CTA's tree 0 (global memory)
    int32_t* err;
    const double* rcp;   // lookup tables (shared memory): 1 / i, sqrt(i), i <= tabn
    const double* sq;
    double gamma, epsilon, c_uct;
    double reward_step, reward_terminal;
    uint32_t k0, k1;     // Philox key
    int64_t tree0;       // global id of the CTA's tree 0
    int32_t tabn, R, puct_f32, ntrees, lpt, po_pad;
    const float* bh; // head biases (shared memory)
    unsigned long long* prof;  // AZG_TREE_PROF builds: per-section cycles of warp 0 (shared memory, no atomics)
};

// a / b for a small integer b through the reciprocal table, without the range checks of div_small (the caller has made them)
__device__ __forceinline__ double div_tab(double a, int b, const double* rcp) {
    const double y = rcp[b];
    const double q = __dmul_rn(a, y);
    const double r = __fma_rn(-q, (double)b, a);
    return __fma_rn(r, y, q);
}
// numerators for which div_tab is the correctly rounded quotient: normal numbers well inside the exponent range (a strict subset of
// div_small's 1e-250 < |a| < 1e250; zero, tiny and non-finite values take the checked form)
__device__ __forceinline__ bool div_tab_ok(double a) {
    const uint32_t e = ((uint32_t)__double2hiint(a) >> 20) & 0x7ffu;
    return (e - 0xC2u) < 0x67Bu;
}

__device__ __forceinline__ void ds_init(const TreeParams& p, const SmTrees& sm, int i, int t) {
    const double* s = p.root_state + (size_t)t * 4;
    double* st = p.dstate + (size_t)t * p.R * 4;
    DRow row;
    row.W[0] = row.W[1] = 0.0;
    row.r = 0.0;
    row.n_e[0] = row.n_e[1] = 0;
    row.prior[0] = row.prior[1] = 0.0f;
    row.V = 0.0f;
    row.node_n = p.root_n_init ? p.root_n_init[t] : 0;
    row.child[0] = row.child[1] = DROW_NONE;
    row.parent = DROW_NONE;
    row.paction = 0;
    row.flags = 0;
    row.pad[0] = row.pad[1] = 0;
    sm.rows[(size_t)i * p.R] = row;
    st[0] = s[0]; st[1] = s[1]; st[2] = s[2]; st[3] = s[3];
    sm.X[i] = make_float4((float)s[0], (float)s[1], (float)s[2], (float)s[3]);
    sm.leaf[i] = 0 | LEAF_EVAL;
    STree z;
    z.n_rows = 1; z.draws = 0; z.levels = 0; z.terms = 0; z.depth = 0;
    sm.st[i] = z;
    p.ctr[(size_t)3 * p.B + t] = 0;  // evaluation counter (the post-processing warps add to it when the search ends)
}

// Philox4x32-10 block of one selection draw (stream 0, block 0; rng_block), word .x, fully unrolled
__device__ __forceinline__ uint32_t philox_draw_x(uint32_t k0, uint32_t k1, uint32_t tree_lo, uint32_t tree_hi, uint32_t idx) {
    uint32_t cx = idx, cy = 0u, cz = tree_lo, cw = tree_hi;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, cx), lo0 = 0xD2511F53u * cx;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, cz), lo1 = 0xCD9E8D57u * cz;
        cx = hi1 ^ cy ^ k0;
        cy = lo1;
        cz = hi0 ^ cw ^ k1;
        cw = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return cx;
}

// The selection rule of one node as a function of its statistics (mcts.py:483-484 + helpers.argmax): bit 0 = arg max of the two PUCT
// scores, bit 1 = the scores are equal (random tie-break), bit 2 = a score is NaN.  Straight-line code: one combined guard in front
// of four reciprocal-table divisions (Markstein); large counts and unusual numerators take the checked forms.
#define DS_DEC_A 1u
#define DS_DEC_TIE 2u
#define DS_DEC_NAN 4u
__device__ __forceinline__ uint32_t ds_decide(const DsCtx& cx, double W0, double W1, int n0, int n1, float pr0, float pr1, float V,
                                              int nn) {  // nn = node.n + 1
    const float cuf = (float)cx.c_uct;
    const double pc0 = cx.puct_f32 ? (double)__fmul_rn(pr0, cuf) : (double)pr0 * cx.c_uct;
    const double pc1 = cx.puct_f32 ? (double)__fmul_rn(pr1, cuf) : (double)pr1 * cx.c_uct;
    double u0, u1;
    if (nn <= cx.tabn && (unsigned)n0 < (unsigned)nn && (unsigned)n1 < (unsigned)nn && (n0 == 0 || div_tab_ok(W0)) && (n1 == 0 || div_tab_ok(W1))) {
        const double sq = cx.sq[nn];
        const double q0 = div_tab(W0, n0 > 0 ? n0 : 1, cx.rcp), q1 = div_tab(W1, n1 > 0 ? n1 : 1, cx.rcp);
        const double e0 = div_tab(sq, n0 + 1, cx.rcp), e1 = div_tab(sq, n1 + 1, cx.rcp);
        u0 = (n0 > 0 ? q0 : (double)V) + pc0 * e0;
        u1 = (n1 > 0 ? q1 : (double)V) + pc1 * e1;
    } else {
        const double sq = sqrt_small(nn, cx.sq, cx.tabn);
        u0 = (n0 > 0 ? div_small(W0, n0, cx.rcp, cx.tabn) : (double)V) + pc0 * div_small(sq, n0 + 1, cx.rcp, cx.tabn);
        u1 = (n1 > 0 ? div_small(W1, n1, cx.rcp, cx.tabn) : (double)V) + pc1 * div_small(sq, n1 + 1, cx.rcp, cx.tabn);
    }
    return (u1 > u0 ? DS_DEC_A : 0u) | (u0 == u1 ? DS_DEC_TIE : 0u) | ((u0 != u0 || u1 != u1) ? DS_DEC_NAN : 0u);
}

// One simulation step of the trees of a WARP on the shared-memory tables: a group of `lpt` consecutive lanes (4 .. 32, a power of two)
// per tree; all 32 lanes call this together (`valid`: this lane's group has a tree, i = its index in the CTA, t = its global id).
//
// ncu on the one-thread-per-tree version (profiles/README.md r2g): ~3200 warp instructions per tree step, issued at ~9 cycles each
// by warps with two active lanes -- the step is bound by the LENGTH of its dependent instruction stream.  This version shortens it:
//   * a node's selection rule (ds_decide) only changes when a backup passes through the node, so it is evaluated THERE, for all
//     levels of the path at once (lane j owns level j), and cached in the row (DRow::pad[0]); the descent reads one 16-byte piece
//     per level (children + cached rule) -- about ten instructions;
//   * the return R = r + gamma R is the only sequential part of the backup: it runs down the levels in registers (the r values come
//     by shuffle), the statistics of all levels are updated in parallel;
//   * the selection draws of the next lpt indices are generated at once, one Philox block per lane, and reduced with two ballots
//     to bit masks (epsilon test / random action per level) -- the generator was 1200 of the 3200 instructions.
// Same arithmetic on the same inputs as d_step: results are bit-identical.
#ifdef AZG_TREE_PROF
#define DSP_BEGIN() long long dsp_last = clock64()
#define DSP_STAMP(k) do { const long long _t = clock64(); if (threadIdx.x == 0) cx.prof[k] += (unsigned long long)(_t - dsp_last); dsp_last = _t; } while (0)
#else
#define DSP_BEGIN()
#define DSP_STAMP(k)
#endif
// shared-memory accesses by 32-bit address: the tables' pointers come out of DsCtx, so the compiler cannot know their address space
__device__ __forceinline__ uint4 ds_lds128(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ double ds_lds64(uint32_t a) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t ds_lds32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t ds_lds16(uint32_t a) {
    uint16_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void ds_sts64(uint32_t a, double v) { asm volatile("st.shared.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory"); }
__device__ __forceinline__ void ds_sts32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void ds_sts16(uint32_t a, uint32_t v) { asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "h"((uint16_t)v) : "memory"); }

__device__ __forceinline__ void ds_step(const DsCtx& cx, const DsCtx* cxs, int i, bool valid, int lane, const bool BACKUP, const bool SELECT) {
    const uint32_t FULL = 0xFFFFFFFFu;
    DSP_BEGIN();
    const SmTrees sm = cx.sm;
    const int lpt = cx.lpt, R = cx.R;
    DRow* rows = sm.rows + (size_t)i * R;
    const uint32_t rows_s = (uint32_t)__cvta_generic_to_shared(rows);                          // row k of this tree at rows_s + 64 k
    const uint32_t path_s = (uint32_t)__cvta_generic_to_shared(sm.path + (size_t)i * R);       // (row << 1 | action) of level k at path_s + 2 k
    const int gl = lane & (lpt - 1), gbase = lane - gl;
    {
        // finish the evaluated row (what the post-processing warp does in the other schedules, mlp.cuh mlp_finish_row): sum the head's
        // four quarter chains in the contract's order, softmax over the two logits, V and priors into the leaf's row.  Done here the
        // evaluation -> post-processing warp -> tree phase hand-over (an mbarrier round trip and a warp wake-up per simulation) is gone.
        // Lanes 0, 1, 2 of the group take V and the two logits (one exponential and one division each instead of two in a row).
        const int leafw = sm.leaf[i];
        const int o = gl < 3 ? gl : 2;
        const int nt = cxs->ntrees, pp = cxs->po_pad;
        const float* part = sm.part + i;
        const float q0 = part[(0 * pp + o) * nt], q1 = part[(1 * pp + o) * nt], q2 = part[(2 * pp + o) * nt], q3 = part[(3 * pp + o) * nt];
        const float out = __fadd_rn(__fadd_rn(__fadd_rn(q0, q1), __fadd_rn(q2, q3)), cxs->bh[o]);
        const float l0 = __shfl_sync(FULL, out, gbase + 1), l1 = __shfl_sync(FULL, out, gbase + 2);
        const float m = l1 > l0 ? l1 : l0;  // softmax_seq over two logits (policies.py:275-297)
        const float e = det::expf_(__fsub_rn(out, m));
        const float e0 = __shfl_sync(FULL, e, gbase + 1), e1 = __shfl_sync(FULL, e, gbase + 2);
        const float sum = __fadd_rn(__fadd_rn(0.0f, e0), e1);
        if (valid && (leafw & LEAF_EVAL) && gl < 3) {
            const uint32_t lrow_s = rows_s + 64u * (uint32_t)(leafw & LEAF_ROW_MASK);
            if (gl == 0) ds_sts32(lrow_s + 40u, __float_as_uint((leafw & LEAF_TERMINAL) ? 0.0f : out));  // mcts.py:406-410
            else ds_sts32(lrow_s + 28u + 4u * gl, __float_as_uint(__fdiv_rn(e, sum)));                   // prior[gl - 1]
        }
    }
    __syncwarp();
    {
        // R = leaf.V; up the path: R = node.r + gamma*R; edge.n += 1; edge.W += R; parent.n += 1 (mcts.py:241-267); then the selection
        // rule of every node whose statistics changed, and of the leaf (whose V and priors the evaluation has just written)
        const int leaf = sm.leaf[i] & LEAF_ROW_MASK;
        const int d = BACKUP ? (int)sm.st[i].depth : 0;
        double Rv = (double)__uint_as_float(ds_lds32(rows_s + 64u * leaf + 40u));
        const double gamma = cx.gamma;
        int hi = valid ? d + 1 : 0;  // items [0, d]: the levels of the path and the leaf
#pragma unroll 1
        while (__any_sync(FULL, hi > 0)) {
            const int lo = hi > lpt ? hi - lpt : 0;
            const int j = lo + gl;  // this lane's item
            const bool act = j < hi, lvl = act && j < d;
            const int e = lvl ? (int)ds_lds16(path_s + 2u * j) : 0;
            const int cj = lvl ? (j + 1 < d ? (int)(ds_lds16(path_s + 2u * j + 2u) >> 1) : leaf) : 0;  // the node level j leads to
            const double rj = ds_lds64(rows_s + 64u * cj + 16u);
            const uint32_t nrow_s = rows_s + 64u * (lvl ? (e >> 1) : leaf);
            const uint4 q0 = ds_lds128(nrow_s), q1 = ds_lds128(nrow_s + 16u), q2 = ds_lds128(nrow_s + 32u);
            const int top = (hi < d ? hi : d) - lo;                  // levels of the path in this chunk
            const int nlev = __reduce_max_sync(FULL, top);           // largest over the warp's groups
            double myR = 0.0;
#pragma unroll 1
            for (int sb = (nlev - 1) & ~3; sb >= 0; sb -= 4) {  // four levels per round: the shuffles do not wait for the chain
                double rq[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) rq[k] = __shfl_sync(FULL, rj, (gbase + sb + k) & 31);
#pragma unroll
                for (int k = 3; k >= 0; --k) {
                    if (sb + k < top) {
                        Rv = rq[k] + gamma * Rv;
                        if (sb + k == gl) myR = Rv;
                    }
                }
            }
            if (act) {
                double W0 = __hiloint2double((int)q0.y, (int)q0.x), W1 = __hiloint2double((int)q0.w, (int)q0.z);
                int n0 = (int)q1.z, n1 = (int)q1.w, nn = (int)q2.w;
                if (lvl) {  // the nodes of a path are distinct: no two lanes touch the same row
                    if (e & 1) { W1 += myR; n1 += 1; ds_sts64(nrow_s + 8u, W1); ds_sts32(nrow_s + 28u, (uint32_t)n1); }
                    else { W0 += myR; n0 += 1; ds_sts64(nrow_s, W0); ds_sts32(nrow_s + 24u, (uint32_t)n0); }
                    nn += 1;
                    ds_sts32(nrow_s + 44u, (uint32_t)nn);
                }
                ds_sts32(nrow_s + 56u, ds_decide(cx, W0, W1, n0, n1, __uint_as_float(q2.x), __uint_as_float(q2.y), __uint_as_float(q2.z), nn + 1));
            }
            hi = lo;
        }
        __syncwarp();
    }
    DSP_STAMP(1);
    if (SELECT) {
        const int64_t tree = cx.tree0 + i;
        const uint32_t k0 = cx.k0, k1 = cx.k1, tlo = (uint32_t)tree, thi = (uint32_t)((uint64_t)tree >> 32);
        const double epsilon = cx.epsilon;
        STree st = sm.st[i];
        const bool eps = epsilon != 0;
        const int dsh = eps ? 1 : 0;             // draws per level = 1 << dsh: random() of epsilon_greedy (if epsilon != 0), then randint / choice
        const int nb = lpt == 32 ? 1 : 2;        // Philox blocks per lane and batch: a batch is nb * lpt <= 32 draws = one 32-bit mask
        const int lpb = (nb * lpt) >> dsh;       // levels served by one batch (a power of two)
        uint32_t RP = 0, RB = 0;                 // per draw of the batch: random() < epsilon; the random action
        int cur = 0, a = -1, levels = 0;
        bool active = valid, expand = false;
        uint32_t nanacc = 0;
        int L = 0;                               // level index, the same for every group of the warp that is still descending
#pragma unroll 1
        while (__any_sync(FULL, active)) {
            const int kb = L & (lpb - 1);
            if (kb == 0) {  // draws st.draws + (L << dsh) + [0, nb * lpt): lane gl generates draws gl and lpt + gl of the batch
                const uint32_t d0 = (uint32_t)(st.draws + (L << dsh) + gl);
                const uint32_t x = philox_draw_x(k0, k1, tlo, thi, d0);
                RP = __ballot_sync(FULL, (double)u32_to_unit(x) < epsilon) >> gbase;
                RB = __ballot_sync(FULL, u32_to_index(x, 2) != 0) >> gbase;
                if (nb == 2) {
                    const uint32_t y = philox_draw_x(k0, k1, tlo, thi, d0 + (uint32_t)lpt);
                    const uint32_t lo_mask = (1u << lpt) - 1u;
                    RP = (RP & lo_mask) | ((__ballot_sync(FULL, (double)u32_to_unit(y) < epsilon) >> gbase) << lpt);
                    RB = (RB & lo_mask) | ((__ballot_sync(FULL, u32_to_index(y, 2) != 0) >> gbase) << lpt);
                }
                if (!eps) RP = 0;
            }
            // one 16-byte piece per level: child[0] | child[1] << 16, parent | paction << 16 | flags << 24, cached rule, -
            const uint4 q3 = ds_lds128(rows_s + 64u * cur + 48u);
            const int sh = kb << dsh;
            const uint32_t rbit = (RB >> (sh + dsh)) & 1u;
            const bool use_r = (((RP >> sh) | (q3.z >> 1)) & 1u) != 0;   // epsilon pick, or equal scores: the random action
            const int an = (int)(use_r ? rbit : (q3.z & DS_DEC_A));
            const int child = (int)(an ? (q3.x >> 16) : (q3.x & 0xFFFFu));
            // branch-free: `term` = the trace ends on an existing terminal node (the root never is one), `go` = this level is descended
            const bool term = ((q3.y >> 24) & ROW_TERMINAL) != 0;
            const bool go = active && !term;
            a = go ? an : (active ? -1 : a);
            nanacc |= go ? q3.z : 0u;
            if (go && gl == 0) ds_sts16(path_s + 2u * L, (uint32_t)((cur << 1) | an));
            levels += go ? 1 : 0;
            expand = expand || (go && child == DROW_NONE);
            active = go && child != DROW_NONE;
            cur = active ? child : cur;
            ++L;
        }
        DSP_STAMP(2);
#ifdef AZG_TREE_PROF
        if (threadIdx.x == 0) cx.prof[7] += (unsigned long long)L;
#endif
        __syncwarp();  // every lane has read the tree's scalars and rows before lane 0 of its group rewrites them
        if (valid && gl == 0) {
            if (nanacc & DS_DEC_NAN) atomicOr(cx.err, ERR_NAN);
            st.draws += levels << dsh;
            st.levels += (uint32_t)levels;
            st.depth = (uint16_t)levels;
            if (expand) {
                const int child = st.n_rows;
                if (child >= R) {
                    atomicOr(cx.err, ERR_CAPACITY);
                    sm.leaf[i] = cur;
                    st.depth = 0;
                } else {
                    st.n_rows = child + 1;
                    const double* sp = cx.dstate + ((size_t)i * R + cur) * 4;
                    const double s[4] = {sp[0], sp[1], sp[2], sp[3]};
                    double o[4], rew;
                    const bool term = env::cartpole_step(s, a, o, rew);
                    // rl/wrappers.py (1.0 / 1.0 without wrappers); read from the shared-memory block here, once per step: as part of the
                    // register copy the two constants cost 20 M sims/s in spills (profiles/README.md r2x)
                    rew = term ? cxs->reward_terminal : cxs->reward_step;
                    double* so = cx.dstate + ((size_t)i * R + child) * 4;
                    so[0] = o[0]; so[1] = o[1]; so[2] = o[2]; so[3] = o[3];
                    DRow nr;
                    nr.W[0] = nr.W[1] = 0.0;
                    nr.r = rew;
                    nr.n_e[0] = nr.n_e[1] = 0;
                    nr.prior[0] = nr.prior[1] = 0.0f;
                    nr.V = 0.0f;
                    nr.node_n = 0;
                    nr.child[0] = nr.child[1] = DROW_NONE;
                    nr.parent = (uint16_t)cur;
                    nr.paction = (uint8_t)a;
                    nr.flags = term ? ROW_TERMINAL : 0;
                    nr.pad[0] = nr.pad[1] = 0;
                    rows[child] = nr;
                    rows[cur].child[a] = (uint16_t)child;
                    sm.X[i] = make_float4((float)o[0], (float)o[1], (float)o[2], (float)o[3]);
                    sm.leaf[i] = child | LEAF_EVAL | (term ? LEAF_TERMINAL : 0);
                }
            } else {
                sm.leaf[i] = cur;
                st.terms += 1;
            }
            sm.st[i] = st;
        }
        __syncwarp();
        DSP_STAMP(4);
    }
}

// The tree phase of the whole-search kernel (qmlp2.cuh TSM): called by every thread of the 16 epilogue warps; mode bit 0 = backup
// of the finished simulation, bit 1 = descent + expansion of the next.  Everything it needs comes out of the DsCtx copy, so the
// level loop holds its addresses in registers (as a NOINLINE function it measured slower: 235 against 295 M sims/s, r2k).
#ifdef AZG_DS_NOINLINE
__device__ __noinline__
#else
__device__ __forceinline__
#endif
void ds_phase(const DsCtx* cxs, int mode) {
    const DsCtx cx = *cxs;
    const int tid = threadIdx.x, lane = tid & 31;
    const int i = tid / cx.lpt, i0 = (tid & ~31) / cx.lpt;  // this lane's tree; the first tree of its warp
    if (i0 >= cx.ntrees) return;  // no tree on this warp
    // lanes without a tree shadow the warp's first tree (they read what its lanes read, at the same points, and write nothing)
    ds_step(cx, cxs, i < cx.ntrees ? i : i0, i < cx.ntrees, lane, (mode & 1) != 0, (mode & 2) != 0);
}

// end of the search: rows in use and per-tree scalars back to the global tables (cooperatively, `nthreads` threads of the CTA)
__device__ __forceinline__ void ds_writeback(const TreeParams& p, const SmTrees& sm, int ntrees, int t0, int tid, int nthreads) {
    const int per_tree = p.R * 4;  // 16-byte pieces per tree
    const uint4* src = reinterpret_cast<const uint4*>(sm.rows);
    uint4* dst = reinterpret_cast<uint4*>(p.drows + (size_t)t0 * p.R);
    for (int k = tid; k < ntrees * per_tree; k += nthreads) {
        const int i = k / per_tree, off = k - i * per_tree;
        if (off < sm.st[i].n_rows * 4) {
            uint4 v = src[k];
            if ((off & 3) == 3) v.z = 0u;  // DRow::pad[0] held the cached selection rule
            dst[k] = v;
        }
    }
    for (int i = tid; i < ntrees; i += nthreads) {
        const STree st = sm.st[i];
        const int t = t0 + i;
        p.n_rows[t] = st.n_rows;
        p.draws[t] = st.draws;
        p.leaf[t] = sm.leaf[i];
        p.ctr[t] = st.levels;
        p.ctr[(size_t)p.B + t] = st.levels * 2;
        p.ctr[(size_t)2 * p.B + t] = st.terms;
        p.ctr[(size_t)3 * p.B + t] = (uint32_t)st.n_rows;  // evaluations: the root and every node created
    }
}

// MCTS.return_results (mcts.py:269-307) for the discrete root
template <class ENV>
__global__ void k_results_discrete(const TreeParams p, int cmax, float* actions, int32_t* counts, double* Q, double* Vt,
                                   int32_t* nchild) {
    constexpr int A = ENV::A;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p.B) return;
    if constexpr (A == 2) {
        const DRow row = load_drow(p.drows + (size_t)t * p.R);
        double q[2];
        for (int a = 0; a < 2; ++a) {
            const int n = row.n_e[a];
            q[a] = n > 0 ? row.W[a] / (double)n : (double)row.V;
            actions[(size_t)t * cmax + a] = (float)a;
            counts[(size_t)t * cmax + a] = n;
            Q[(size_t)t * cmax + a] = q[a];
        }
        nchild[t] = 2;
        double v;
        if (p.v_target == 1) {  // on_policy: np.sum((counts / np.sum(counts)) * Q), n < 8 -> sequential sum from 0.
            const double tot = (double)(row.n_e[0] + row.n_e[1]);
            v = 0.0;
            v += ((double)row.n_e[0] / tot) * q[0];
            v += ((double)row.n_e[1] / tot) * q[1];
        } else {
            v = q[1] > q[0] ? q[1] : q[0];
        }
        Vt[t] = v;
    } else {
        D3Row row;
        load_line0(&row, reinterpret_cast<const D3Row*>(p.drows) + (size_t)t * p.R);
        double q[A];
        for (int a = 0; a < A; ++a) {
            const int n = row.n_e[a];
            q[a] = n > 0 ? row.W[a] / (double)n : (double)row.V;
            actions[(size_t)t * cmax + a] = (float)a;
            counts[(size_t)t * cmax + a] = n;
            Q[(size_t)t * cmax + a] = q[a];
        }
        nchild[t] = A;
        double v;
        if (p.v_target == 1) {  // on_policy: np.sum((counts / np.sum(counts)) * Q), n < 8 -> sequential sum from 0.
            int tot = 0;
            for (int a = 0; a < A; ++a) tot += row.n_e[a];
            v = 0.0;
            for (int a = 0; a < A; ++a) v += ((double)row.n_e[a] / (double)tot) * q[a];
        } else {  // Q.max()
            v = q[0];
            for (int a = 1; a < A; ++a) v = q[a] > v ? q[a] : v;
        }
        Vt[t] = v;
    }
}

// engine.cu -- C ABI (include/azg.h) and kernel orchestration of the batched MCTS engine.
//
// One search = init -> evaluate(root) -> [continuous: root widening insert] ->
//              N x { step<backup of previous sim, select, expand> -> evaluate(leaves) } -> final backup.
// Trees are independent, so there is no inter-CTA synchronisation anywhere.  Two schedules, identical results: the whole search as
// ONE persistent kernel per chunk of trees (AZG_FLAG_FUSED, qmlp2.cuh: default with the tensor-core evaluation), or 2N+3 launches
// captured once into a CUDA graph per (B, n_rollouts, tape, tree_id0) and replayed.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <map>
#include <string>
#include <tuple>
#include <type_traits>
#include <utility>
#include <vector>

#include "../../include/azg.h"
#include "common.cuh"
#include "env.cuh"
#include "mlp.cuh"
#include "qmlp.cuh"
#include "qmlp2.cuh"
#include "search_wg.cuh"
#include "selfplay.cuh"
#include "tree_continuous.cuh"
#include "tree_discrete.cuh"

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
#define CK(call)                                                                                             \
    do {                                                                                                     \
        cudaError_t _e = (call);                                                                             \
        if (_e != cudaSuccess)                                                                               \
            return fail(AZG_ECUDA, std::string(#call) + ": " + cudaGetErrorString(_e) + " (" __FILE__ ":" +  \
                                       std::to_string(__LINE__) + ")");                                      \
    } while (0)

struct azg_engine {
    azg_config cfg;
    int R = 0, HS = 0, P = 0, PO_PAD = 0, cmax = 0, K3 = 0;
    int64_t n_weights = 0;
    int wcount = 0;
    size_t mlp_smem = 0;
    int sm_count = 0;
    // device memory
    DRow* drows = nullptr;
    double* dstate = nullptr;
    CRow* crows = nullptr;
    CHot* et = nullptr;
    uint4* ctl = nullptr;  // [4][max_trees] chunk planes of the control blocks (common.cuh)
    float* chead = nullptr;
    int32_t *pw_table = nullptr, *n_rows = nullptr, *draws = nullptr, *leaf = nullptr;
    uint8_t* path = nullptr;
    uint32_t* mt = nullptr;     // AZG_FLAG_RNG_MT19937: [B][625]
    uint32_t* tmt = nullptr;    // AZG_FLAG_RNG_MT19937, continuous: torch's generator [B][628]
    uint16_t* dpath = nullptr;  // discrete: recorded path of the current simulation [B][R]
    int32_t* ddepth = nullptr;
    uint32_t* ctr = nullptr;
    float4* X = nullptr;
    double* root_state = nullptr;
    int32_t* root_n_init = nullptr;
    int32_t* err = nullptr;
    float* wpack = nullptr;
    uint64_t* d_seed = nullptr;  // Philox key read by the kernels (azg_set_seed)
    unsigned long long* stats = nullptr;  // cycle accounting of the whole-search kernel (azg_fused_stats)
    double* dtab = nullptr;      // rcp_tab[AZG_TAB + 1], sqrt_tab[AZG_TAB + 1] (common.cuh div_small)
    // AZG_FLAG_EVAL_Q8: int8 digit planes + f32 side table of the tensor-core evaluation kernel (qmlp.cuh)
    int8_t* qdigits = nullptr;
    int8_t* qdigits_nat = nullptr;  // rows in natural order (search_wg.cuh)
    int fused_mode = 0;             // 0: whole-search kernel chosen by batch size; 1: two-phase (qmlp2.cuh); 2: warpgroups (search_wg.cuh)
    size_t wg_smem = 0;
    float* qfl = nullptr;
    int qfl_count = 0;
    size_t qmlp_smem = 0;
    double reward_step = 1.0, reward_terminal = 1.0;  // azg_set_reward_model (rl/wrappers.py around the searched env)
    int last_fused_kind = 0;        // whole-search kernel of the last search: 1 two-phase, 2 warpgroups, 3 two-phase with the trees in shared memory
    size_t smem_optin = 0;
    size_t tsm_smem_max = 0;        // discrete whole-search kernel with the trees in shared memory (qmlp2.cuh TSM): dynamic shared memory it may use
    bool q8 = false;
    // continuous tree: root edge tables + control blocks in ONE allocation, pinned in L2 (persisting access-policy window on every
    // launch that walks trees): they are touched by every simulation of every tree (37.7 MB at 65536 trees, against 126 MB of L2),
    // while the row tables stream through
    void* hot_block = nullptr;
    size_t hot_bytes = 0;
    cudaLaunchAttribute l2attr;
    int l2_on = 0;
    bool fused = false;  // AZG_FLAG_FUSED: the whole continuous search in one persistent kernel (qmlp2.cuh)
    bool mcc = false;    // AZG_FLAG_ENV_MOUNTAIN_CAR_CONTINUOUS: the continuous kernels are instantiated for env::MountainCarContinuous
    bool mc = false;     // AZG_FLAG_ENV_MOUNTAIN_CAR: the discrete kernels are instantiated for env::MountainCar (three-action rows)
    bool ac = false;     // AZG_FLAG_ENV_ACROBOT: the discrete kernels are instantiated for env::Acrobot (three-action rows, 6 inputs)
    // results staging (device) + pinned host staging for the *_host entry point
    float* r_actions = nullptr;
    int32_t* r_counts = nullptr;
    double* r_Q = nullptr;
    double* r_Vt = nullptr;
    int32_t* r_nchild = nullptr;
    void* h_pinned = nullptr;
    size_t h_pinned_bytes = 0;
    // azg_search_host_begin / _end: a second set of result buffers, a copy stream and per-slot events, so that the D2H of one search's
    // results overlaps the next search
    float* r2_actions = nullptr;
    int32_t* r2_counts = nullptr;
    double* r2_Q = nullptr;
    double* r2_Vt = nullptr;
    int32_t* r2_nchild = nullptr;
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_done[2] = {nullptr, nullptr}, ev_copied[2] = {nullptr, nullptr};
    int32_t* h_err = nullptr;  // pinned, one word per slot
    bool pending[2] = {false, false};
    cudaStream_t own_stream = nullptr;
    // tapes
    const float *tapeV = nullptr, *tapeP = nullptr, *tapeA = nullptr;
    bool weights_set = false;
    // last search
    int last_B = 0, last_N = 0;
    int64_t launches = 0;
    std::map<std::tuple<int, int, int>, cudaGraphExec_t> graphs;  // (B, n_rollouts, tape)
    int64_t tree_word = 0;  // value of d_seed[1] (global id of tree 0 for graph-captured launches)
};

static int head_dim_of(const azg_config& c) {
    if (c.variant == AZG_DISCRETE) return c.num_actions;
    return c.num_components > 1 ? 3 * c.num_components : 2;
}

// width of the hidden-state arrays the host hands in and gets back: CartPole and Acrobot 4, MountainCar and the continuous envs 2
static int state_width(const azg_engine* e) { return e->cfg.variant == AZG_DISCRETE && !e->mc ? 4 : 2; }

static int pw_limit(double c_pw, double kappa, int n) { return (int)std::ceil(c_pw * std::pow((double)(n + 1), kappa)); }

extern "C" const char* azg_last_error(void) { return g_err.c_str(); }
extern "C" const char* azg_version(void) { return "azg 0.1 (sm_100a)"; }

template <typename T>
static cudaError_t dalloc(T** p, size_t n) {
    return cudaMalloc((void**)p, n * sizeof(T));
}

static cudaError_t launch_mlp(const azg_engine* e, const MlpParams& m, cudaStream_t st, bool set_attr);

extern "C" void azg_destroy(azg_engine* e) {
    if (!e) return;
    cudaSetDevice(e->cfg.device);
    for (auto& kv : e->graphs) cudaGraphExecDestroy(kv.second);
    void* ptrs[] = {e->drows, e->dstate, e->crows, e->hot_block, e->chead, e->pw_table, e->n_rows, e->draws,
                    e->leaf, e->path, e->dpath, e->ddepth, e->mt, e->tmt, e->ctr, e->X, e->root_state, e->root_n_init, e->err, e->wpack, e->d_seed, e->stats, e->dtab, e->qdigits, e->qdigits_nat, e->qfl, e->r_actions,
                    e->r_counts, e->r_Q, e->r_Vt, e->r_nchild};
    for (void* q : ptrs)
        if (q) cudaFree(q);
    if (e->h_pinned) cudaFreeHost(e->h_pinned);
    if (e->h_err) cudaFreeHost(e->h_err);
    for (void* q : {(void*)e->r2_actions, (void*)e->r2_counts, (void*)e->r2_Q, (void*)e->r2_Vt, (void*)e->r2_nchild})
        if (q) cudaFree(q);
    for (int k = 0; k < 2; ++k) {
        if (e->ev_done[k]) cudaEventDestroy(e->ev_done[k]);
        if (e->ev_copied[k]) cudaEventDestroy(e->ev_copied[k]);
    }
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    if (e->own_stream) cudaStreamDestroy(e->own_stream);
    delete e;
}

extern "C" int azg_create(const azg_config* cfg, azg_engine** out) {
    if (!cfg || !out) return fail(AZG_EINVAL, "null argument");
    *out = nullptr;
    const azg_config& c = *cfg;
    if (c.variant != AZG_DISCRETE && c.variant != AZG_CONTINUOUS) return fail(AZG_EINVAL, "variant must be AZG_DISCRETE or AZG_CONTINUOUS");
    if (c.max_rollouts < 1 || c.max_trees < 1) return fail(AZG_EINVAL, "max_rollouts and max_trees must be >= 1");
    if (c.hidden != 128 && c.hidden != 64) return fail(AZG_EINVAL, "hidden width must be 64 or 128 (weights are staged in shared memory)");
    if (c.n_hidden < 1 || c.n_hidden > 4) return fail(AZG_EINVAL, "n_hidden must be in 1..4");
    if (c.activation < AZG_ACT_RELU || c.activation > AZG_ACT_HARDSWISH) return fail(AZG_EINVAL, "activation must be one of AZG_ACT_*");
    if ((c.flags & AZG_FLAG_EVAL_Q8) && c.activation > AZG_ACT_ELU)
        return fail(AZG_EINVAL, "AZG_FLAG_EVAL_Q8 serves relu and elu (the configured activations); the others run on the FP32 kernel");
    const bool mcc = (c.flags & AZG_FLAG_ENV_MOUNTAIN_CAR_CONTINUOUS) != 0;
    if (mcc && (c.variant != AZG_CONTINUOUS || c.state_dim != 2))
        return fail(AZG_EINVAL, "AZG_FLAG_ENV_MOUNTAIN_CAR_CONTINUOUS needs the continuous variant and state_dim 2");
    const bool mc = (c.flags & AZG_FLAG_ENV_MOUNTAIN_CAR) != 0;
    if (mc && mcc) return fail(AZG_EINVAL, "AZG_FLAG_ENV_MOUNTAIN_CAR and AZG_FLAG_ENV_MOUNTAIN_CAR_CONTINUOUS exclude each other");
    if (mc && (c.variant != AZG_DISCRETE || c.num_actions != 3 || c.state_dim != 2))
        return fail(AZG_EINVAL, "AZG_FLAG_ENV_MOUNTAIN_CAR needs the discrete variant, num_actions 3 and state_dim 2");
    const bool ac = (c.flags & AZG_FLAG_ENV_ACROBOT) != 0;
    if (ac && (mc || mcc)) return fail(AZG_EINVAL, "AZG_FLAG_ENV_ACROBOT excludes both MountainCar flags");
    if (ac && (c.variant != AZG_DISCRETE || c.num_actions != 3 || c.state_dim != 6))
        return fail(AZG_EINVAL, "AZG_FLAG_ENV_ACROBOT needs the discrete variant, num_actions 3 and state_dim 6");
    if (c.variant == AZG_DISCRETE) {
        if (!mc && !ac && (c.num_actions != 2 || c.state_dim != 4))
            return fail(AZG_EINVAL, "discrete variant is CartPole (num_actions 2, state_dim 4) or, with AZG_FLAG_ENV_MOUNTAIN_CAR, MountainCar-v0 "
                                    "(num_actions 3, state_dim 2) or, with AZG_FLAG_ENV_ACROBOT, Acrobot-v1 (num_actions 3, state_dim 6)");
        if (c.max_rollouts + 2 > 65534) return fail(AZG_EINVAL, "max_rollouts too large for 16-bit child links");
        if ((mc || ac) && c.max_rollouts + 2 > 16384)
            return fail(AZG_EINVAL, "MountainCar-v0 and Acrobot-v1 support max_rollouts <= 16382 (a path entry holds row << 2 | action in 16 bits)");
    } else {
        if (!mcc && c.state_dim != 3) return fail(AZG_EINVAL, "continuous variant is Pendulum: state_dim must be 3");
        if (c.num_components < 1 || c.num_components > AZG_MAX_K) return fail(AZG_EINVAL, "num_components must be in 1..8");
        if (c.max_rollouts + 2 > 255) return fail(AZG_EINVAL, "continuous variant supports n_rollouts <= 253 (8-bit row links)");
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(AZG_ECUDA, "no CUDA device: the engine has no CPU fallback");
    if (c.device < 0 || c.device >= ndev) return fail(AZG_EINVAL, "bad device ordinal");
    CK(cudaSetDevice(c.device));
    azg_engine* e = new azg_engine();
    e->cfg = c;
    e->mcc = mcc;
    e->mc = mc;
    e->ac = ac;
    e->R = c.max_rollouts + 2;
    e->P = head_dim_of(c);
    e->PO_PAD = ((1 + e->P) + 3) / 4 * 4;
    e->K3 = 3 * (c.num_components > 0 ? c.num_components : 1);
    e->HS = (e->K3 + 3) / 4 * 4;
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, c.device));
    e->sm_count = prop.multiProcessorCount;
    e->smem_optin = (size_t)prop.sharedMemPerBlockOptin;
    const int H = c.hidden;
    int64_t nw = (int64_t)c.state_dim * H + H;
    for (int l = 1; l < c.n_hidden; ++l) nw += (int64_t)H * H + H;
    nw += H + 1 + (int64_t)e->P * H + e->P;
    e->n_weights = nw;
    e->wcount = c.state_dim * H + H + (c.n_hidden - 1) * (H * H + H) + H * e->PO_PAD + e->PO_PAD;
    e->mlp_smem = ((size_t)e->wcount + (size_t)MLP_NGRP * (H + e->PO_PAD) * MLP_UNIT) * sizeof(float);
    if (e->mlp_smem > (size_t)prop.sharedMemPerBlockOptin) {
        delete e;
        return fail(AZG_EINVAL, "network does not fit in shared memory");
    }
    e->q8 = (c.flags & AZG_FLAG_EVAL_Q8) != 0;
    if (e->q8) {
        e->qfl_count = (c.state_dim * H + H + (c.n_hidden - 1) * 2 * H + H * e->PO_PAD + e->PO_PAD + 3) / 4 * 4;
        e->qmlp_smem = qmlp2_smem_bytes(c.n_hidden - 1, e->qfl_count, (c.flags & AZG_FLAG_FUSED) != 0);
        e->wg_smem = search_wg_smem_bytes(c.n_hidden - 1, e->qfl_count);
        // AZG_FUSED_KERNEL=two_phase | warpgroups forces one whole-search kernel (experiments); default: by batch size (launch_fused_t)
        const char* fk = getenv("AZG_FUSED_KERNEL");
        e->fused_mode = !fk ? 0 : (fk[0] == 't' ? 1 : 2);
        if (getenv("AZG_FUSED_V1")) e->fused_mode = 1;
        if (H != 128 || c.n_hidden < 2 || c.n_hidden > 3 || e->PO_PAD > Q2_MAX_PO || e->qmlp_smem > (size_t)prop.sharedMemPerBlockOptin ||
            prop.major != 10) {
            delete e;
            return fail(AZG_EINVAL, "AZG_FLAG_EVAL_Q8 needs hidden = 128, n_hidden in {2, 3}, at most 15 head outputs and an sm_100 device (tcgen05)");
        }
    }
    e->fused = (c.flags & AZG_FLAG_FUSED) != 0;
    if ((c.flags & AZG_FLAG_RNG_MT19937) && c.variant == AZG_CONTINUOUS && e->fused) {
        delete e;
        return fail(AZG_EINVAL, "AZG_FLAG_RNG_MT19937 with the continuous search runs one launch per simulation (no AZG_FLAG_FUSED)");
    }
    if (e->fused && !(e->q8 && c.state_dim == (c.variant == AZG_CONTINUOUS ? (mcc ? 2 : 3) : (mc ? 2 : (ac ? 6 : 4))))) {
        delete e;
        return fail(AZG_EINVAL, "AZG_FLAG_FUSED needs AZG_FLAG_EVAL_Q8 and the shipped envs (state_dim 3 Pendulum / 2 MountainCarContinuous / 4 CartPole / "
                                "2 MountainCar / 6 Acrobot)");
    }
    const size_t B = c.max_trees, R = e->R;
    std::vector<int32_t> pwt;
    if (c.variant == AZG_CONTINUOUS) {
        int cm = 1;
        for (int n = 0; n < c.max_rollouts + 2; ++n) {
            pwt.push_back(pw_limit(c.c_pw, c.kappa, n));
            if (n <= c.max_rollouts) cm = std::max(cm, pwt.back());
        }
        e->cmax = cm + 1;
        if (cm > CROW_MAX_KIDS) {
            delete e;
            return fail(AZG_ECAPACITY, "progressive-widening fan-out exceeds the 15 inline child slots of a row (c_pw/kappa/n_rollouts too large)");
        }
    } else {
        e->cmax = c.num_actions;
    }
#define ALLOC(ptr, n)                                   \
    do {                                                \
        cudaError_t _e = dalloc(&e->ptr, (n));          \
        if (_e != cudaSuccess) {                        \
            std::string m = cudaGetErrorString(_e);     \
            azg_destroy(e);                             \
            return fail(AZG_ECUDA, "cudaMalloc " #ptr ": " + m); \
        }                                               \
    } while (0)
    if (c.variant == AZG_DISCRETE) {
        ALLOC(drows, B * R * (mc || ac ? sizeof(D3Row) / sizeof(DRow) : 1));  // MountainCar, Acrobot: D3Row [B][R]
        ALLOC(dstate, B * R * 4);
        ALLOC(dpath, B * R);
        ALLOC(ddepth, B);
        if (c.flags & AZG_FLAG_RNG_MT19937) ALLOC(mt, B * (MT_N + 1));
    } else {
        ALLOC(crows, B * R);
        {
            e->hot_bytes = B * (CROOT_MAX_KIDS * sizeof(CHot) + sizeof(CCtl));
            char* hb = nullptr;
            cudaError_t _e = cudaMalloc(&hb, e->hot_bytes);
            if (_e != cudaSuccess) {
                std::string m = cudaGetErrorString(_e);
                azg_destroy(e);
                return fail(AZG_ECUDA, "cudaMalloc hot block: " + m);
            }
            e->hot_block = hb;
            e->et = reinterpret_cast<CHot*>(hb);
            e->ctl = reinterpret_cast<uint4*>(hb + B * CROOT_MAX_KIDS * sizeof(CHot));
            const size_t persist_max = (size_t)std::max(0, prop.persistingL2CacheMaxSize), win_max = (size_t)std::max(0, prop.accessPolicyMaxWindowSize);
            if (persist_max > 0 && win_max > 0 && !getenv("AZG_NO_L2_PERSIST")) {
                const size_t want = std::min(persist_max, e->hot_bytes);
                size_t have = 0;
                cudaDeviceGetLimit(&have, cudaLimitPersistingL2CacheSize);
                if (have < want) cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want);
                cudaDeviceGetLimit(&have, cudaLimitPersistingL2CacheSize);
                memset(&e->l2attr, 0, sizeof e->l2attr);
                e->l2attr.id = cudaLaunchAttributeAccessPolicyWindow;
                cudaAccessPolicyWindow& w = e->l2attr.val.accessPolicyWindow;
                w.base_ptr = hb;
                w.num_bytes = std::min(e->hot_bytes, win_max);
                w.hitRatio = (float)std::min(1.0, (double)have / (double)w.num_bytes);
                w.hitProp = cudaAccessPropertyPersisting;
                w.missProp = cudaAccessPropertyStreaming;
                e->l2_on = have > 0;
                cudaGetLastError();
            }
        }
        ALLOC(chead, B * R * e->HS);
        ALLOC(pw_table, pwt.size());
        ALLOC(path, B * R);
        if (c.flags & AZG_FLAG_RNG_MT19937) {  // CPython's and torch's generator per tree
            ALLOC(mt, B * (MT_N + 1));
            ALLOC(tmt, B * TMT_WORDS);
        }
        CK(cudaMemcpy(e->pw_table, pwt.data(), pwt.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
        CK(cudaMemset(e->chead, 0, B * R * e->HS * sizeof(float)));
    }
    ALLOC(n_rows, B); ALLOC(draws, B); ALLOC(leaf, B);
    ALLOC(ctr, 4 * B);
    ALLOC(X, B * (ac ? env::Acrobot::XW : 1));  // Acrobot: 6 inputs in two float4 per tree
    ALLOC(root_state, B * 4);
    ALLOC(root_n_init, B);
    ALLOC(err, 1);
    ALLOC(wpack, (size_t)e->wcount);
    ALLOC(d_seed, 2);  // Philox key, global id of tree 0 for graph-captured launches
    ALLOC(stats, 16);
    ALLOC(dtab, 2 * (AZG_TAB + 1));
    if (e->q8) {
        ALLOC(qdigits, (size_t)(c.n_hidden - 1) * 3 * QMLP_PLANE);
        ALLOC(qdigits_nat, (size_t)(c.n_hidden - 1) * 3 * QMLP_PLANE);
        ALLOC(qfl, (size_t)e->qfl_count);
    }
    ALLOC(r_actions, B * e->cmax); ALLOC(r_counts, B * e->cmax); ALLOC(r_Q, B * e->cmax); ALLOC(r_Vt, B); ALLOC(r_nchild, B);
#undef ALLOC
    CK(cudaMemset(e->err, 0, sizeof(int32_t)));
    CK(cudaMemset(e->stats, 0, 16 * sizeof(unsigned long long)));
    CK(cudaMemset(e->d_seed, 0, 2 * sizeof(uint64_t)));
    CK(cudaMemcpy(e->d_seed, &c.seed, sizeof(uint64_t), cudaMemcpyHostToDevice));
    {
        std::vector<double> tab(2 * (AZG_TAB + 1), 0.0);
        for (int i = 1; i <= AZG_TAB; ++i) {
            volatile double di = (double)i;
            tab[i] = 1.0 / di;                      // IEEE division: correctly rounded
            tab[AZG_TAB + 1 + i] = std::sqrt(di);   // IEEE sqrt: correctly rounded
        }
        CK(cudaMemcpy(e->dtab, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice));
    }
    CK(cudaMemset(e->n_rows, 0, B * sizeof(int32_t)));
    CK(cudaMemset(e->ctr, 0, 4 * B * sizeof(uint32_t)));
    {
        MlpParams dummy;
        memset(&dummy, 0, sizeof dummy);
        CK(launch_mlp(e, dummy, nullptr, true));
    }
    e->h_pinned_bytes = B * 4 * sizeof(double) + B * sizeof(int32_t) +
                        B * e->cmax * (sizeof(float) + sizeof(int32_t) + sizeof(double)) + B * (sizeof(double) + sizeof(int32_t)) + 256;
    CK(cudaMallocHost(&e->h_pinned, e->h_pinned_bytes));
    CK(cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking));
    *out = e;
    return AZG_OK;
}

extern "C" int64_t azg_num_weights(const azg_engine* e) { return e ? e->n_weights : 0; }
extern "C" int32_t azg_cmax(const azg_engine* e) { return e ? e->cmax : 0; }
extern "C" int32_t azg_rows(const azg_engine* e) { return e ? e->R : 0; }
extern "C" int32_t azg_head_dim(const azg_engine* e) {
    if (!e) return 0;
    return e->cfg.variant == AZG_DISCRETE ? e->cfg.num_actions : e->K3;
}

// state_dict order -> packed k-major layout consumed by k_mlp
static void pack_weights(const azg_engine* e, const float* w, std::vector<float>& out) {
    const int H = e->cfg.hidden, S = e->cfg.state_dim, L = e->cfg.n_hidden, P = e->P, PO = e->PO_PAD;
    out.assign(e->wcount, 0.0f);
    float* d = out.data();
    for (int l = 0; l < L; ++l) {
        const int K = l == 0 ? S : H;
        for (int j = 0; j < H; ++j)
            for (int k = 0; k < K; ++k) d[(size_t)k * H + j] = w[(size_t)j * K + k];
        d += (size_t)K * H;
        w += (size_t)K * H;
        memcpy(d, w, H * sizeof(float));
        d += H;
        w += H;
    }
    const float* wv = w;            // value_head.weight [1][H]
    const float* bv = w + H;        // value_head.bias [1]
    const float* wd = w + H + 1;    // dist_head.weight [P][H]
    const float* bd = wd + (size_t)P * H;
    for (int k = 0; k < H; ++k) {
        d[(size_t)k * PO] = wv[k];
        for (int q = 0; q < P; ++q) d[(size_t)k * PO + 1 + q] = wd[(size_t)q * H + k];
    }
    d += (size_t)H * PO;
    d[0] = bv[0];
    for (int q = 0; q < P; ++q) d[1 + q] = bd[q];
}

// AZG_FLAG_EVAL_Q8 packing (contract: oracle/azg_oracle.h "AZO_EVAL_Q8"; consumer: qmlp.cuh).  Hidden layer l >= 1, output j:
// e = clamp(biased_exponent(max_k |W[j][k]| * 1.004f), 32, 200); Wq = rni(W * 2^(149-e)); balanced base-256 digits = bytes of
// (Wq + 0x8080) ^ 0x8080; planes (hi, mid, lo) in the UMMA K-major canonical layout [k/16][j][16]; cw[j] = 2^(e-133).
static void pack_weights_q8(const azg_engine* e, const float* w, std::vector<int8_t>& digits, std::vector<float>& fl, bool natural_rows = false) {
    const int H = e->cfg.hidden, S = e->cfg.state_dim, L = e->cfg.n_hidden, P = e->P, PO = e->PO_PAD;
    digits.assign((size_t)(L - 1) * 3 * QMLP_PLANE, 0);
    fl.assign(e->qfl_count, 0.0f);
    float* d = fl.data();
    for (int j = 0; j < H; ++j)
        for (int k = 0; k < S; ++k) d[(size_t)k * H + j] = w[(size_t)j * S + k];
    d += (size_t)S * H;
    w += (size_t)S * H;
    memcpy(d, w, H * sizeof(float));
    d += H;
    w += H;
    auto bits = [](float f) { uint32_t u; memcpy(&u, &f, 4); return u; };
    auto from_bits = [](uint32_t u) { float f; memcpy(&f, &u, 4); return f; };
    for (int l = 1; l < L; ++l) {
        int8_t* pl = digits.data() + (size_t)(l - 1) * 3 * QMLP_PLANE;
        for (int j = 0; j < H; ++j) {
            float wmax = 0.0f;
            for (int k = 0; k < H; ++k) wmax = fmaxf(wmax, fabsf(w[(size_t)j * H + k]));
            volatile float scaled = wmax * 1.004f;
            int ex = (int)((bits(scaled) >> 23) & 0xFF);
            ex = ex < 32 ? 32 : (ex > 200 ? 200 : ex);
            const float sc = from_bits((uint32_t)(276 - ex) << 23);
            d[2 * j] = from_bits((uint32_t)(ex - 6) << 23);
            d[2 * j + 1] = w[(size_t)H * H + j];
            for (int k = 0; k < H; ++k) {
                volatile float tq = w[(size_t)j * H + k] * sc;
                const float tv = tq;
                int32_t q = tv != tv ? 0 : (tv >= 2147483648.0f ? INT32_MAX : (tv <= -2147483648.0f ? INT32_MIN : (int32_t)nearbyintf(tv)));
                const uint32_t t = ((uint32_t)q + 0x8080u) ^ 0x8080u;
                if (natural_rows) {  // search_wg.cuh: [k/16][step of 16 outputs][plane][16 rows][16 B]
                    const size_t o = (size_t)(k / 16) * WG_B_KCHUNK + (size_t)(j / 16) * WG_B_STEP + (size_t)(j % 16) * 16 + (k % 16);
                    pl[o] = (int8_t)((t >> 16) & 0xFF);
                    pl[o + 256] = (int8_t)((t >> 8) & 0xFF);
                    pl[o + 512] = (int8_t)(t & 0xFF);
                    continue;
                }
                const size_t o = (size_t)(k / 16) * 2048 + (size_t)qmlp_perm_row(j) * 16 + (k % 16);
                pl[o] = (int8_t)((t >> 16) & 0xFF);
                pl[QMLP_PLANE + o] = (int8_t)((t >> 8) & 0xFF);
                pl[2 * QMLP_PLANE + o] = (int8_t)(t & 0xFF);
            }
        }
        d += 2 * H;
        w += (size_t)H * H + H;
    }
    const float* wv = w;
    const float* bv = w + H;
    const float* wd = w + H + 1;
    const float* bd = wd + (size_t)P * H;
    for (int k = 0; k < H; ++k) {
        d[(size_t)k * PO] = wv[k];
        for (int q = 0; q < P; ++q) d[(size_t)k * PO + 1 + q] = wd[(size_t)q * H + k];
    }
    d += (size_t)H * PO;
    d[0] = bv[0];
    for (int q = 0; q < P; ++q) d[1 + q] = bd[q];
}

extern "C" int azg_set_weights(azg_engine* e, const float* flat, int64_t n, void* stream) {
    if (!e || !flat) return fail(AZG_EINVAL, "null argument");
    if (n != e->n_weights) return fail(AZG_EINVAL, "weight count " + std::to_string(n) + " != expected " + std::to_string(e->n_weights));
    CK(cudaSetDevice(e->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    std::vector<float> host(n);
    cudaPointerAttributes at;
    bool on_device = cudaPointerGetAttributes(&at, flat) == cudaSuccess && (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged);
    cudaGetLastError();
    if (on_device) {
        CK(cudaMemcpyAsync(host.data(), flat, n * sizeof(float), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    } else {
        memcpy(host.data(), flat, n * sizeof(float));
    }
    std::vector<float> packed;
    pack_weights(e, host.data(), packed);
    CK(cudaMemcpyAsync(e->wpack, packed.data(), packed.size() * sizeof(float), cudaMemcpyHostToDevice, st));
    std::vector<int8_t> qd;
    std::vector<float> qf;
    if (e->q8) {
        pack_weights_q8(e, host.data(), qd, qf);
        CK(cudaMemcpyAsync(e->qdigits, qd.data(), qd.size(), cudaMemcpyHostToDevice, st));
        std::vector<int8_t> qn;
        std::vector<float> qf2;
        pack_weights_q8(e, host.data(), qn, qf2, true);
        CK(cudaMemcpyAsync(e->qdigits_nat, qn.data(), qn.size(), cudaMemcpyHostToDevice, st));
        CK(cudaStreamSynchronize(st));  // qn is a local
        CK(cudaMemcpyAsync(e->qfl, qf.data(), qf.size() * sizeof(float), cudaMemcpyHostToDevice, st));
    }
    CK(cudaStreamSynchronize(st));
    e->weights_set = true;
    return AZG_OK;
}

extern "C" int azg_set_tapes(azg_engine* e, const float* d_V, const float* d_prior, const float* d_action) {
    if (!e) return fail(AZG_EINVAL, "null engine");
    if (d_V) {
        if (e->cfg.variant == AZG_DISCRETE && !d_prior) return fail(AZG_EINVAL, "discrete tapes need priors");
        if (e->cfg.variant == AZG_CONTINUOUS && !d_action) return fail(AZG_EINVAL, "continuous tapes need actions");
    }
    e->tapeV = d_V;
    e->tapeP = d_V ? d_prior : nullptr;
    e->tapeA = d_V ? d_action : nullptr;
    return AZG_OK;
}

static TreeParams make_params(const azg_engine* e, int B, int64_t tree_id0) {
    TreeParams p;
    memset(&p, 0, sizeof p);
    const azg_config& c = e->cfg;
    p.B = B; p.R = e->R; p.A = c.num_actions; p.K = c.num_components; p.HS = e->HS;
    p.puct_f32 = c.puct_f32; p.v_target = c.v_target; p.use_tape = e->tapeV != nullptr;
    p.c_uct = c.c_uct; p.gamma = c.gamma; p.epsilon = c.epsilon;
    p.reward_step = e->reward_step; p.reward_terminal = e->reward_terminal;
    p.gamma_f32 = (float)c.gamma; p.action_bound = c.action_bound;
    p.seedp = e->d_seed; p.tree_id0 = tree_id0;
    p.drows = e->drows; p.dstate = e->dstate;
    p.crows = e->crows; p.et = e->et; p.ctl = e->ctl; p.BS = e->cfg.max_trees; p.chead = e->chead;
    p.pw_table = e->pw_table;
    p.rcp_tab = e->dtab; p.sqrt_tab = e->dtab + AZG_TAB + 1;
    p.n_rows = e->n_rows; p.draws = e->draws; p.leaf = e->leaf; p.path = e->path; p.dpath = e->dpath; p.ddepth = e->ddepth; p.mt = e->mt; p.tmt = e->tmt; p.rng_mt = e->mt != nullptr;
    p.ctr = e->ctr; p.X = e->X; p.root_state = e->root_state; p.root_n_init = e->root_n_init; p.err = e->err;
    p.tapeV = e->tapeV; p.tapeP = e->tapeP; p.tapeA = e->tapeA;
    p.prof = e->stats + 8;
    return p;
}

static MlpParams make_mlp_params(const azg_engine* e, int n) {
    MlpParams m;
    memset(&m, 0, sizeof m);
    const azg_config& c = e->cfg;
    m.wpack = e->wpack; m.wcount = e->wcount; m.L = c.n_hidden; m.P = e->P; m.PO_PAD = e->PO_PAD;
    m.n = n; m.X = reinterpret_cast<const float*>(e->X); m.xstride = e->ac ? 4 * env::Acrobot::XW : 4; m.mode = 0;
    m.variant = c.variant; m.A = c.num_actions; m.K = c.num_components; m.R = e->R; m.HS = e->HS;
    m.ls_min = c.log_std_min; m.ls_max = c.log_std_max;
    m.leaf = e->leaf; m.drows = e->drows; m.crows = e->crows; m.chead = e->chead; m.evals = e->ctr + (size_t)3 * n;
    m.ctl = e->ctl; m.et = e->et; m.BS = c.max_trees; m.gamma_f32 = (float)c.gamma;
    m.head_dim = azg_head_dim(e);
    m.qdigits = e->qdigits; m.qdigits_nat = e->qdigits_nat; m.qfl = e->qfl; m.qfl_count = e->qfl_count;
    m.stats = e->stats;
    return m;
}

// kernel launch carrying the persisting-L2 window of the hot block (recorded into graph nodes under stream capture)
template <typename... KArgs, typename... Args>
static cudaError_t launch_ex(const azg_engine* e, void (*kernel)(KArgs...), int grid, int block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cfg.attrs = const_cast<cudaLaunchAttribute*>(&e->l2attr);
    cfg.numAttrs = e->l2_on ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

template <int H, int S, int ACT>
static cudaError_t launch_mlp_t(const azg_engine* e, const MlpParams& m, cudaStream_t st, bool set_attr) {
    if (set_attr) return cudaFuncSetAttribute(k_mlp<H, S, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e->mlp_smem);
    const int units = (m.n + MLP_UNIT - 1) / MLP_UNIT;
    const int grid = std::max(1, std::min((units + MLP_NGRP - 1) / MLP_NGRP, e->sm_count));
    return launch_ex(e, k_mlp<H, S, ACT>, grid, MLP_THREADS(H), e->mlp_smem, st, m);
}

// ENV (env.cuh) selects the tree and env of the whole-search kernels; the evaluation-only launch reads ENV::S (layer 0) alone
template <class ENV, int ACT, int NL>
static cudaError_t launch_qmlp_t(const azg_engine* e, const MlpParams& m, cudaStream_t st, bool set_attr) {
    if (set_attr) {
        cudaError_t ce = cudaFuncSetAttribute(k_qmlp2<ENV, ACT, NL, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e->qmlp_smem);
        if (ce != cudaSuccess) return ce;
        ce = cudaFuncSetAttribute(k_qmlp2<ENV, ACT, NL, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e->qmlp_smem);
        if (ce != cudaSuccess) return ce;
        if constexpr (env::actions_of<ENV>() == 2) {  // trees in shared memory (CartPole): everything the SM has beyond the kernel's static allocation
            cudaFuncAttributes fa;
            ce = cudaFuncGetAttributes(&fa, k_qmlp2<ENV, ACT, NL, true, true>);
            if (ce != cudaSuccess) return ce;
            const_cast<azg_engine*>(e)->tsm_smem_max = e->smem_optin - std::min(e->smem_optin, fa.sharedSizeBytes);
            ce = cudaFuncSetAttribute(k_qmlp2<ENV, ACT, NL, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e->tsm_smem_max);
            if (ce != cudaSuccess) return ce;
        }
        // search_wg.cuh raises its 16 tree + evaluation warps to 104 registers with setmaxnreg: the CTA's pool (640 threads x the
        // kernel's register count) must hold 512 x 104 + 128 x 56, or the instruction would wait forever
        cudaFuncAttributes fa;
        ce = cudaFuncGetAttributes(&fa, k_search_wg<ENV, ACT, NL>);
        if (ce != cudaSuccess) return ce;
        if (fa.numRegs * WG_THREADS < WG_EPI_THREADS * WG_EPI_REGS + 128 * WG_MMA_REGS) return cudaErrorLaunchOutOfResources;
        return cudaFuncSetAttribute(k_search_wg<ENV, ACT, NL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e->wg_smem);
    }
    const int grid = std::max(1, std::min((m.n + 127) / 128, e->sm_count));
    TreeParams none;
    memset(&none, 0, sizeof none);
    return launch_ex(e, k_qmlp2<ENV, ACT, NL, false>, grid, Q2_THREADS, e->qmlp_smem, st, m, none, 0, 0, 0);
}

// whole-search kernel (AZG_FLAG_FUSED): one persistent launch per chunk of at most sm_count x Q2_MAX_TILES x 128 trees
template <class ENV, int ACT, int NL>
static cudaError_t launch_fused_t(const azg_engine* e, const MlpParams& m, const TreeParams& p, int N, cudaStream_t st, int* launches) {
    int chunk = e->sm_count * Q2_MAX_TILES * 128;
    if constexpr (env::actions_of<ENV>() == 2) {
        // CartPole search: up to two full waves of shared-memory-resident trees (cap per SM x SMs each) beat the two-phase kernel on
        // rows in HBM, whose simulation takes 32 us whatever the batch (measured, profiles/README.md r2p: 8192 trees 248 M sims/s
        // there against 2 x 4096 at 337 M) -- so such a batch is cut into equal chunks, one launch each
        int cap = 0;
        while (cap < 128 && qmlp2_tsm_smem_bytes(NL, e->qfl_count, cap + 1, p.R, e->PO_PAD) <= e->tsm_smem_max) ++cap;
        const long long wave = (long long)cap * e->sm_count;
        if (cap > 0 && !p.rng_mt && !getenv("AZG_NO_TSM") && e->fused_mode != 2 && p.B > wave && p.B <= 2 * wave) chunk = (p.B + 1) / 2;
    }
    for (int lo = 0; lo < p.B; lo += chunk) {
        const int hi = std::min(p.B, lo + chunk);
        cudaError_t ce;
        // Which whole-search kernel: measured on B200 (profiles/README.md r2c, trees per GPU -> M sims/s, Pendulum N = 100):
        //   two-phase (qmlp2.cuh)     8192: 332   16384: 641   32768: 934   65536: 1056   131072:  962
        //   warpgroups (search_wg)    8192: 155   16384: 292   32768: 571   65536: 1113   131072: 1050
        // A warpgroup evaluates its tile alone (one thread per row, all 128 columns), so a simulation never takes less than ~52 us;
        // in the two-phase kernel 16 warps share a tile and a thin batch finishes a simulation in ~24 us.  From about three full
        // tiles per SM on, the independent warpgroups win (the tree step of one hides under the evaluation of the others).
        const bool two_phase = e->fused_mode == 1 || (e->fused_mode == 0 && (hi - lo) < 3 * 128 * e->sm_count);
        // Discrete search, thin batch: when the rows of ceil(trees / SMs) trees fit in an SM's shared memory next to the evaluation's
        // operands, the CTA keeps its trees there for the whole search (tree_discrete.cuh ds_step; BASELINE config 3: 28 trees per SM)
        int tsm_per = 0;
        if constexpr (env::actions_of<ENV>() == 2) {  // (not built for three-action rows: MountainCar's thin batches run the two-phase kernel)
            const int per = (hi - lo + e->sm_count - 1) / e->sm_count;
            if (two_phase && !p.rng_mt && !getenv("AZG_NO_TSM") && per <= 128 &&
                qmlp2_tsm_smem_bytes(NL, e->qfl_count, per, p.R, e->PO_PAD) <= e->tsm_smem_max)
                tsm_per = per;
        }
        const_cast<azg_engine*>(e)->last_fused_kind = tsm_per ? 3 : (two_phase ? 1 : 2);
        if (tsm_per) {
            if constexpr (env::actions_of<ENV>() == 2) {
                const int grid = (hi - lo + tsm_per - 1) / tsm_per;
                ce = launch_ex(e, k_qmlp2<ENV, ACT, NL, true, true>, grid, Q2_THREADS, qmlp2_tsm_smem_bytes(NL, e->qfl_count, tsm_per, p.R, e->PO_PAD), st, m, p, N, lo, hi);
            }
        } else if (two_phase) {
            const int grid = std::max(1, std::min((hi - lo + 127) / 128, e->sm_count));
            ce = launch_ex(e, k_qmlp2<ENV, ACT, NL, true>, grid, Q2_THREADS, e->qmlp_smem, st, m, p, N, lo, hi);
        } else {
            // four warpgroups per CTA, each with its own tile: small batches are spread over every SM (a CTA's trees over its four
            // warpgroups), large ones use all SMs with up to WG_MAX_ROUNDS x 4 tiles each
            const int grid = std::max(1, std::min((hi - lo + 3) / 4, e->sm_count));
            ce = launch_ex(e, k_search_wg<ENV, ACT, NL>, grid, WG_THREADS, e->wg_smem, st, m, p, N, lo, hi);
        }
        ++*launches;
        if (ce != cudaSuccess) return ce;
    }
    return cudaSuccess;
}

// The S of the CartPole / Pendulum tables below names the env (azg_create: state_dim 4 is CartPole, 3 Pendulum); MountainCarContinuous
// has tables of its own, selected by its flag (their instantiations run in tests/test_mountain_car_gpu.py)
template <int S>
using ShippedEnv = std::conditional_t<S == 4, env::CartPole, env::Pendulum>;

static cudaError_t launch_fused(const azg_engine* e, const MlpParams& m, const TreeParams& p, int N, cudaStream_t st, int* launches) {
    const int S = e->cfg.state_dim, A = e->cfg.activation, NL = e->cfg.n_hidden - 1;
    if (e->ac) {
#define FUSED_AC_CASE(a, nl) \
    if (A == a && NL == nl) return launch_fused_t<env::Acrobot, a, nl>(e, m, p, N, st, launches);
        FUSED_AC_CASE(0, 1) FUSED_AC_CASE(1, 1) FUSED_AC_CASE(0, 2) FUSED_AC_CASE(1, 2)
#undef FUSED_AC_CASE
        return cudaErrorInvalidValue;
    }
    if (e->mc) {
#define FUSED_MC_CASE(a, nl) \
    if (A == a && NL == nl) return launch_fused_t<env::MountainCar, a, nl>(e, m, p, N, st, launches);
        FUSED_MC_CASE(0, 1) FUSED_MC_CASE(1, 1) FUSED_MC_CASE(0, 2) FUSED_MC_CASE(1, 2)
#undef FUSED_MC_CASE
        return cudaErrorInvalidValue;
    }
    if (e->mcc) {
#define FUSED_MCC_CASE(a, nl) \
    if (A == a && NL == nl) return launch_fused_t<env::MountainCarContinuous, a, nl>(e, m, p, N, st, launches);
        FUSED_MCC_CASE(0, 1) FUSED_MCC_CASE(1, 1) FUSED_MCC_CASE(0, 2) FUSED_MCC_CASE(1, 2)
#undef FUSED_MCC_CASE
        return cudaErrorInvalidValue;
    }
#define FUSED_CASE(s, a, nl) \
    if (S == s && A == a && NL == nl) return launch_fused_t<ShippedEnv<s>, a, nl>(e, m, p, N, st, launches);
    FUSED_CASE(3, 0, 1) FUSED_CASE(3, 1, 1) FUSED_CASE(3, 0, 2) FUSED_CASE(3, 1, 2)
    FUSED_CASE(4, 0, 1) FUSED_CASE(4, 1, 1) FUSED_CASE(4, 0, 2) FUSED_CASE(4, 1, 2)
#undef FUSED_CASE
    return cudaErrorInvalidValue;
}

static cudaError_t launch_mlp(const azg_engine* e, const MlpParams& m, cudaStream_t st, bool set_attr) {
    const int H = e->cfg.hidden, S = e->cfg.state_dim, A = e->cfg.activation;
    if (e->q8) {
        const int NL = e->cfg.n_hidden - 1;
        if (e->ac) {
#define QMLP_AC_CASE(a, nl) \
    if (A == a && NL == nl) return launch_qmlp_t<env::Acrobot, a, nl>(e, m, st, set_attr);
            QMLP_AC_CASE(0, 1) QMLP_AC_CASE(1, 1) QMLP_AC_CASE(0, 2) QMLP_AC_CASE(1, 2)
#undef QMLP_AC_CASE
            return cudaErrorInvalidValue;
        }
        if (e->mc) {
#define QMLP_MC_CASE(a, nl) \
    if (A == a && NL == nl) return launch_qmlp_t<env::MountainCar, a, nl>(e, m, st, set_attr);
            QMLP_MC_CASE(0, 1) QMLP_MC_CASE(1, 1) QMLP_MC_CASE(0, 2) QMLP_MC_CASE(1, 2)
#undef QMLP_MC_CASE
            return cudaErrorInvalidValue;
        }
        if (e->mcc) {
#define QMLP_MCC_CASE(a, nl) \
    if (A == a && NL == nl) return launch_qmlp_t<env::MountainCarContinuous, a, nl>(e, m, st, set_attr);
            QMLP_MCC_CASE(0, 1) QMLP_MCC_CASE(1, 1) QMLP_MCC_CASE(0, 2) QMLP_MCC_CASE(1, 2)
#undef QMLP_MCC_CASE
            return cudaErrorInvalidValue;
        }
#define QMLP_CASE(s, a, nl) \
    if (S == s && A == a && NL == nl) return launch_qmlp_t<ShippedEnv<s>, a, nl>(e, m, st, set_attr);
        QMLP_CASE(4, 0, 1) QMLP_CASE(4, 1, 1) QMLP_CASE(3, 0, 1) QMLP_CASE(3, 1, 1)
        QMLP_CASE(4, 0, 2) QMLP_CASE(4, 1, 2) QMLP_CASE(3, 0, 2) QMLP_CASE(3, 1, 2)
#undef QMLP_CASE
        return cudaErrorInvalidValue;
    }
    if (e->ac) {  // layer 0 with six inputs (Acrobot)
#define MLP_AC_CASE(h, a) \
    if (H == h && A == a) return launch_mlp_t<h, 6, a>(e, m, st, set_attr);
        MLP_AC_CASE(128, 0) MLP_AC_CASE(128, 1) MLP_AC_CASE(128, 2) MLP_AC_CASE(128, 3) MLP_AC_CASE(128, 4) MLP_AC_CASE(128, 5)
        MLP_AC_CASE(64, 0) MLP_AC_CASE(64, 1) MLP_AC_CASE(64, 2) MLP_AC_CASE(64, 3) MLP_AC_CASE(64, 4) MLP_AC_CASE(64, 5)
#undef MLP_AC_CASE
        return cudaErrorInvalidValue;
    }
    if (e->mcc || e->mc) {  // layer 0 with two inputs (both MountainCar envs; k_mlp reads the row layout at run time)
#define MLP_MCC_CASE(h, a) \
    if (H == h && A == a) return launch_mlp_t<h, 2, a>(e, m, st, set_attr);
        MLP_MCC_CASE(128, 0) MLP_MCC_CASE(128, 1) MLP_MCC_CASE(128, 2) MLP_MCC_CASE(128, 3) MLP_MCC_CASE(128, 4) MLP_MCC_CASE(128, 5)
        MLP_MCC_CASE(64, 0) MLP_MCC_CASE(64, 1) MLP_MCC_CASE(64, 2) MLP_MCC_CASE(64, 3) MLP_MCC_CASE(64, 4) MLP_MCC_CASE(64, 5)
#undef MLP_MCC_CASE
        return cudaErrorInvalidValue;
    }
#define MLP_CASE(h, s, a) \
    if (H == h && S == s && A == a) return launch_mlp_t<h, s, a>(e, m, st, set_attr);
    MLP_CASE(128, 4, 0) MLP_CASE(128, 4, 1) MLP_CASE(128, 3, 0) MLP_CASE(128, 3, 1)
    MLP_CASE(64, 4, 0) MLP_CASE(64, 4, 1) MLP_CASE(64, 3, 0) MLP_CASE(64, 3, 1)
    MLP_CASE(128, 4, 2) MLP_CASE(128, 4, 3) MLP_CASE(128, 4, 4) MLP_CASE(128, 4, 5)
    MLP_CASE(128, 3, 2) MLP_CASE(128, 3, 3) MLP_CASE(128, 3, 4) MLP_CASE(128, 3, 5)
    MLP_CASE(64, 4, 2) MLP_CASE(64, 4, 3) MLP_CASE(64, 4, 4) MLP_CASE(64, 4, 5)
    MLP_CASE(64, 3, 2) MLP_CASE(64, 3, 3) MLP_CASE(64, 3, 4) MLP_CASE(64, 3, 5)
#undef MLP_CASE
    return cudaErrorInvalidValue;
}

template <bool BK, bool SEL>
static cudaError_t launch_step_discrete(const azg_engine* e, const TreeParams& p, cudaStream_t st) {
    if (e->mc) return launch_ex(e, k_step_discrete<env::MountainCar, BK, SEL>, (p.B + 127) / 128, 128, 0, st, p);
    if (e->ac) return launch_ex(e, k_step_discrete<env::Acrobot, BK, SEL>, (p.B + 127) / 128, 128, 0, st, p);
    return launch_ex(e, k_step_discrete<env::CartPole, BK, SEL>, (p.B + 127) / 128, 128, 0, st, p);
}

template <bool BK, bool SEL>
static cudaError_t launch_step_continuous(const azg_engine* e, const TreeParams& p, cudaStream_t st) {
    if (e->mcc) return launch_ex(e, k_step_continuous<env::MountainCarContinuous, BK, SEL>, (p.B + 127) / 128, 128, 0, st, p);
    return launch_ex(e, k_step_continuous<env::Pendulum, BK, SEL>, (p.B + 127) / 128, 128, 0, st, p);
}

// per-launch CUDA-event timing used by azg_profile_search (classes: 0 tree step, 1 evaluation, 2 setup)
struct Prof {
    std::vector<cudaEvent_t> ev;  // start/stop pairs
    std::vector<int> cls;
};

// enqueue the whole search on `st`; returns the number of kernels launched
static int enqueue_search(azg_engine* e, int B, int N, int64_t tree_id0, cudaStream_t st, cudaError_t* cerr, Prof* prof = nullptr, bool tree_word = false) {
    TreeParams p = make_params(e, B, tree_word ? 0 : tree_id0);
    p.tree_word = tree_word ? 1 : 0;
    const MlpParams m = make_mlp_params(e, B);
    const bool tape = p.use_tape != 0;
    int launches = 0;
    cudaError_t ce = cudaSuccess;
    auto begin = [&](int cls) {
        if (!prof) return;
        cudaEvent_t a, b;
        cudaEventCreate(&a);
        cudaEventCreate(&b);
        prof->ev.push_back(a);
        prof->ev.push_back(b);
        prof->cls.push_back(cls);
        cudaEventRecord(a, st);
    };
    auto end = [&]() {
        if (prof) cudaEventRecord(prof->ev.back(), st);
    };
#define LK(cls, expr)                                   \
    do {                                                \
        begin(cls);                                     \
        expr;                                           \
        end();                                          \
        ++launches;                                     \
        if (ce == cudaSuccess) ce = cudaGetLastError(); \
    } while (0)
    const int tb = 128, tg = (B + tb - 1) / tb;
    if (e->fused && !tape && !prof) {  // the whole search in one persistent kernel per chunk of trees (qmlp2.cuh, FUSED)
        ce = launch_fused(e, m, p, N, st, &launches);
        *cerr = ce;
        return launches;
    }
    if (e->cfg.variant == AZG_DISCRETE) {
        if (e->mc) LK(2, (k_init_discrete<env::MountainCar><<<tg, tb, 0, st>>>(p)));
        else if (e->ac) LK(2, (k_init_discrete<env::Acrobot><<<tg, tb, 0, st>>>(p)));
        else LK(2, (k_init_discrete<env::CartPole><<<tg, tb, 0, st>>>(p)));
        if (!tape) LK(1, ce = launch_mlp(e, m, st, false));
        for (int it = 0; it < N; ++it) {
            if (it == 0) LK(0, ce = (launch_step_discrete<false, true>(e, p, st)));
            else LK(0, ce = (launch_step_discrete<true, true>(e, p, st)));
            if (!tape) LK(1, ce = launch_mlp(e, m, st, false));
        }
        LK(0, ce = (launch_step_discrete<true, false>(e, p, st)));
    } else {
        if (e->mcc) LK(2, (k_init_continuous<env::MountainCarContinuous><<<tg, tb, 0, st>>>(p)));
        else LK(2, (k_init_continuous<env::Pendulum><<<tg, tb, 0, st>>>(p)));
        if (!tape) LK(1, ce = launch_mlp(e, m, st, false));
        LK(2, (k_root_insert_continuous<<<tg, tb, 0, st>>>(p)));
        for (int it = 0; it < N; ++it) {
            if (it == 0) LK(0, ce = (launch_step_continuous<false, true>(e, p, st)));
            else LK(0, ce = (launch_step_continuous<true, true>(e, p, st)));
            if (!tape) LK(1, ce = launch_mlp(e, m, st, false));
        }
        LK(0, ce = (launch_step_continuous<true, false>(e, p, st)));
    }
#undef LK
    *cerr = ce;
    return launches;
}

static int run_search(azg_engine* e, int B, const double* d_root_state, const int32_t* d_root_n_init, int N, int64_t tree_id0,
                      cudaStream_t st) {
    if (!e) return fail(AZG_EINVAL, "null engine");
    if (B < 1 || B > e->cfg.max_trees) return fail(AZG_EINVAL, "B out of range (max_trees = " + std::to_string(e->cfg.max_trees) + ")");
    if (N < 1 || N > e->cfg.max_rollouts) return fail(AZG_EINVAL, "n_rollouts out of range (max_rollouts = " + std::to_string(e->cfg.max_rollouts) + ")");
    if (!d_root_state) return fail(AZG_EINVAL, "null root state");
    if (!e->weights_set && !e->tapeV) return fail(AZG_EINVAL, "azg_set_weights has not been called");
    CK(cudaSetDevice(e->cfg.device));
    const int sd = state_width(e);
    // stage the roots in engine-owned buffers so the captured graph has fixed addresses
    if (d_root_state != e->root_state)
        CK(cudaMemcpyAsync(e->root_state, d_root_state, (size_t)B * sd * sizeof(double), cudaMemcpyDeviceToDevice, st));
    if (e->cfg.variant == AZG_DISCRETE) {
        if (d_root_n_init) {
            if (d_root_n_init != e->root_n_init)
                CK(cudaMemcpyAsync(e->root_n_init, d_root_n_init, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        } else {
            CK(cudaMemsetAsync(e->root_n_init, 0, (size_t)B * sizeof(int32_t), st));
        }
    }
    cudaError_t ce = cudaSuccess;
    if ((e->cfg.flags & AZG_FLAG_NO_GRAPH) || (e->fused && !e->tapeV)) {  // the fused search is one launch per chunk: nothing to capture
        e->launches = enqueue_search(e, B, N, tree_id0, st, &ce);
        if (ce != cudaSuccess) return fail(AZG_ECUDA, std::string("kernel launch: ") + cudaGetErrorString(ce));
    } else {
        const int tape = e->tapeV != nullptr;
        const auto key = std::make_tuple(B, N, tape);  // tree_id0 is read from device memory (TreeParams::tree_word): one graph serves every id
        auto it = e->graphs.find(key);
        if (it == e->graphs.end() || tape) {  // tape pointers may change between calls: always re-capture
            if (it != e->graphs.end()) {
                cudaGraphExecDestroy(it->second);
                e->graphs.erase(it);
            }
            cudaGraph_t g = nullptr;
            CK(cudaStreamBeginCapture(e->own_stream, cudaStreamCaptureModeThreadLocal));
            const int n = enqueue_search(e, B, N, tree_id0, e->own_stream, &ce, nullptr, true);
            cudaError_t ee = cudaStreamEndCapture(e->own_stream, &g);
            if (ce != cudaSuccess || ee != cudaSuccess) {
                if (g) cudaGraphDestroy(g);
                return fail(AZG_ECUDA, std::string("graph capture: ") + cudaGetErrorString(ce != cudaSuccess ? ce : ee));
            }
            cudaGraphExec_t ge = nullptr;
            cudaError_t ie = cudaGraphInstantiate(&ge, g, 0);
            cudaGraphDestroy(g);
            if (ie != cudaSuccess) return fail(AZG_ECUDA, std::string("graph instantiate: ") + cudaGetErrorString(ie));
            if (e->graphs.size() > 32) {
                for (auto& kv : e->graphs) cudaGraphExecDestroy(kv.second);
                e->graphs.clear();
            }
            e->graphs[key] = ge;
            e->launches = n;
            it = e->graphs.find(key);
        }
        e->launches = 2 * (int64_t)N + 3 + (e->cfg.variant == AZG_CONTINUOUS ? 1 : 0) - (tape ? N + 1 : 0);
        if (e->tree_word != tree_id0) {
            k_set_seed<<<1, 1, 0, st>>>(e->d_seed + 1, (uint64_t)tree_id0);
            CK(cudaGetLastError());
            e->tree_word = tree_id0;
        }
        CK(cudaGraphLaunch(it->second, st));
    }
    e->last_B = B;
    e->last_N = N;
    return AZG_OK;
}

extern "C" int azg_search_discrete(azg_engine* e, int32_t B, const double* d_root_state, const int32_t* d_root_n_init,
                                   int32_t n_rollouts, int64_t tree_id0, void* stream) {
    if (e && e->cfg.variant != AZG_DISCRETE) return fail(AZG_EINVAL, "engine was created for the continuous variant");
    return run_search(e, B, d_root_state, d_root_n_init, n_rollouts, tree_id0, (cudaStream_t)stream);
}

extern "C" int azg_search_continuous(azg_engine* e, int32_t B, const double* d_root_state, int32_t n_rollouts, int64_t tree_id0,
                                     void* stream) {
    if (e && e->cfg.variant != AZG_CONTINUOUS) return fail(AZG_EINVAL, "engine was created for the discrete variant");
    return run_search(e, B, d_root_state, nullptr, n_rollouts, tree_id0, (cudaStream_t)stream);
}

extern "C" int azg_profile_search(azg_engine* e, int32_t B, const double* d_root_state, const int32_t* d_root_n_init,
                                  int32_t n_rollouts, int64_t tree_id0, void* stream, float ms_out[3], int32_t launches_out[3]) {
    if (!e || !d_root_state || !ms_out || !launches_out) return fail(AZG_EINVAL, "null argument");
    if (B < 1 || B > e->cfg.max_trees) return fail(AZG_EINVAL, "B out of range");
    if (n_rollouts < 1 || n_rollouts > e->cfg.max_rollouts) return fail(AZG_EINVAL, "n_rollouts out of range");
    if (!e->weights_set && !e->tapeV) return fail(AZG_EINVAL, "azg_set_weights has not been called");
    CK(cudaSetDevice(e->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    const int sd = state_width(e);
    if (d_root_state != e->root_state)
        CK(cudaMemcpyAsync(e->root_state, d_root_state, (size_t)B * sd * sizeof(double), cudaMemcpyDeviceToDevice, st));
    if (e->cfg.variant == AZG_DISCRETE) {
        if (d_root_n_init) CK(cudaMemcpyAsync(e->root_n_init, d_root_n_init, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        else CK(cudaMemsetAsync(e->root_n_init, 0, (size_t)B * sizeof(int32_t), st));
    }
    Prof prof;
    cudaError_t ce = cudaSuccess;
    e->launches = enqueue_search(e, B, n_rollouts, tree_id0, st, &ce, &prof);
    cudaError_t se = cudaStreamSynchronize(st);
    for (int k = 0; k < 3; ++k) { ms_out[k] = 0.0f; launches_out[k] = 0; }
    for (size_t i = 0; i < prof.cls.size(); ++i) {
        float ms = 0.0f;
        if (cudaEventElapsedTime(&ms, prof.ev[2 * i], prof.ev[2 * i + 1]) == cudaSuccess) {
            ms_out[prof.cls[i]] += ms;
            launches_out[prof.cls[i]] += 1;
        }
    }
    for (cudaEvent_t ev : prof.ev) cudaEventDestroy(ev);
    if (ce != cudaSuccess) return fail(AZG_ECUDA, std::string("kernel launch: ") + cudaGetErrorString(ce));
    if (se != cudaSuccess) return fail(AZG_ECUDA, std::string("sync: ") + cudaGetErrorString(se));
    e->last_B = B;
    e->last_N = n_rollouts;
    return AZG_OK;
}

extern "C" int azg_root_results(azg_engine* e, int32_t B, float* d_actions, int32_t* d_counts, double* d_Q, double* d_V_target,
                                int32_t* d_n_children, void* stream) {
    if (!e || !d_actions || !d_counts || !d_Q || !d_V_target || !d_n_children) return fail(AZG_EINVAL, "null argument");
    if (B < 1 || B > e->cfg.max_trees) return fail(AZG_EINVAL, "B out of range");
    CK(cudaSetDevice(e->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    const TreeParams p = make_params(e, B, 0);
    const int tb = 128, tg = (B + tb - 1) / tb;
    if (e->cfg.variant == AZG_DISCRETE && e->mc) k_results_discrete<env::MountainCar><<<tg, tb, 0, st>>>(p, e->cmax, d_actions, d_counts, d_Q, d_V_target, d_n_children);
    else if (e->cfg.variant == AZG_DISCRETE && e->ac) k_results_discrete<env::Acrobot><<<tg, tb, 0, st>>>(p, e->cmax, d_actions, d_counts, d_Q, d_V_target, d_n_children);
    else if (e->cfg.variant == AZG_DISCRETE) k_results_discrete<env::CartPole><<<tg, tb, 0, st>>>(p, e->cmax, d_actions, d_counts, d_Q, d_V_target, d_n_children);
    else k_results_continuous<<<tg, tb, 0, st>>>(p, e->cmax, d_actions, d_counts, d_Q, d_V_target, d_n_children);
    CK(cudaGetLastError());
    return AZG_OK;
}

extern "C" int azg_status(azg_engine* e, void* stream) {
    if (!e) return fail(AZG_EINVAL, "null engine");
    CK(cudaSetDevice(e->cfg.device));
    int32_t h = 0;
    CK(cudaMemcpyAsync(&h, e->err, sizeof h, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CK(cudaStreamSynchronize((cudaStream_t)stream));
    if (h) CK(cudaMemsetAsync(e->err, 0, sizeof h, (cudaStream_t)stream));
    if (h & ERR_NAN) return fail(AZG_ENAN, "NaN in a UCT vector (helpers.py:47-48)");
    if (h & ERR_CAPACITY) return fail(AZG_ECAPACITY, "tree arena or child fan-out capacity exceeded");
    if (h & ERR_WRAP) return fail(AZG_EWRAP, "Acrobot-v1: an angle needed more than 64 iterations of wrap (gym would loop on)");
    return AZG_OK;
}

extern "C" int azg_search_host(azg_engine* e, int32_t B, const double* h_root_state, const int32_t* h_root_n_init, int32_t n_rollouts,
                               int64_t tree_id0, float* h_actions, int32_t* h_counts, double* h_Q, double* h_V_target,
                               int32_t* h_n_children) {
    if (!e || !h_root_state || !h_actions || !h_counts || !h_Q || !h_V_target || !h_n_children) return fail(AZG_EINVAL, "null argument");
    if (B < 1 || B > e->cfg.max_trees) return fail(AZG_EINVAL, "B out of range");
    if (e->cfg.variant == AZG_CONTINUOUS && h_root_n_init) return fail(AZG_EINVAL, "root_n_init is a discrete-only argument");
    CK(cudaSetDevice(e->cfg.device));
    cudaStream_t st = e->own_stream;
    const int sd = state_width(e);
    const size_t cm = e->cmax;
    // carve the pinned staging buffer
    char* hp = (char*)e->h_pinned;
    double* p_root = (double*)hp; hp += (size_t)B * 4 * sizeof(double);
    double* p_Q = (double*)hp; hp += (size_t)B * cm * sizeof(double);
    double* p_Vt = (double*)hp; hp += (size_t)B * sizeof(double);
    float* p_act = (float*)hp; hp += (size_t)B * cm * sizeof(float);
    int32_t* p_cnt = (int32_t*)hp; hp += (size_t)B * cm * sizeof(int32_t);
    int32_t* p_nc = (int32_t*)hp; hp += (size_t)B * sizeof(int32_t);
    int32_t* p_rn = (int32_t*)hp;
    {
        cudaPointerAttributes at;
        const bool root_pinned = cudaPointerGetAttributes(&at, h_root_state) == cudaSuccess && at.type == cudaMemoryTypeHost;
        cudaGetLastError();
        if (!root_pinned) memcpy(p_root, h_root_state, (size_t)B * sd * sizeof(double));
        CK(cudaMemcpyAsync(e->root_state, root_pinned ? h_root_state : p_root, (size_t)B * sd * sizeof(double), cudaMemcpyHostToDevice, st));
    }
    const int32_t* d_rn = nullptr;
    if (h_root_n_init) {
        memcpy(p_rn, h_root_n_init, (size_t)B * sizeof(int32_t));
        CK(cudaMemcpyAsync(e->root_n_init, p_rn, (size_t)B * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        d_rn = e->root_n_init;
    }
    int rc = run_search(e, B, e->root_state, d_rn, n_rollouts, tree_id0, st);
    if (rc) return rc;
    rc = azg_root_results(e, B, e->r_actions, e->r_counts, e->r_Q, e->r_Vt, e->r_nchild, st);
    if (rc) return rc;
    // Output buffers that are page-locked (cudaHostAlloc / cudaHostRegister / torch pin_memory) receive the results by DMA
    // directly; pageable ones go through the engine's pinned staging buffer and one host memcpy each.
    auto pinned = [](const void* h) {
        cudaPointerAttributes at;
        const bool ok = cudaPointerGetAttributes(&at, h) == cudaSuccess && at.type == cudaMemoryTypeHost;
        cudaGetLastError();
        return ok;
    };
    const bool direct = pinned(h_actions) && pinned(h_counts) && pinned(h_Q) && pinned(h_V_target) && pinned(h_n_children);
    CK(cudaMemcpyAsync(direct ? h_actions : p_act, e->r_actions, (size_t)B * cm * sizeof(float), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(direct ? h_counts : p_cnt, e->r_counts, (size_t)B * cm * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(direct ? h_Q : p_Q, e->r_Q, (size_t)B * cm * sizeof(double), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(direct ? h_V_target : p_Vt, e->r_Vt, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(direct ? h_n_children : p_nc, e->r_nchild, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    rc = azg_status(e, st);  // synchronises
    if (!direct) {
        memcpy(h_actions, p_act, (size_t)B * cm * sizeof(float));
        memcpy(h_counts, p_cnt, (size_t)B * cm * sizeof(int32_t));
        memcpy(h_Q, p_Q, (size_t)B * cm * sizeof(double));
        memcpy(h_V_target, p_Vt, (size_t)B * sizeof(double));
        memcpy(h_n_children, p_nc, (size_t)B * sizeof(int32_t));
    }
    return rc;
}

// Pipelined form of azg_search_host: begin(slot) enqueues H2D of the roots, the search, the result extraction and -- on a copy stream --
// the D2H of the results, and returns at once; end(slot) waits until that slot's results are in the caller's buffers.  With two slots
// in flight the PCIe transfer of search i (13 MB at 65536 trees) runs under search i + 1.  Every host buffer must be page-locked.
extern "C" int azg_search_host_begin(azg_engine* e, int32_t slot, int32_t B, const double* h_root_state, const int32_t* h_root_n_init,
                                     int32_t n_rollouts, int64_t tree_id0, float* h_actions, int32_t* h_counts, double* h_Q,
                                     double* h_V_target, int32_t* h_n_children) {
    if (!e || !h_root_state || !h_actions || !h_counts || !h_Q || !h_V_target || !h_n_children) return fail(AZG_EINVAL, "null argument");
    if (slot < 0 || slot > 1) return fail(AZG_EINVAL, "slot must be 0 or 1");
    if (B < 1 || B > e->cfg.max_trees) return fail(AZG_EINVAL, "B out of range");
    if (e->cfg.variant == AZG_CONTINUOUS && h_root_n_init) return fail(AZG_EINVAL, "root_n_init is a discrete-only argument");
    if (e->pending[slot]) return fail(AZG_EINVAL, "slot is still in flight: call azg_search_host_end first");
    CK(cudaSetDevice(e->cfg.device));
    auto pinned = [](const void* h) {
        cudaPointerAttributes at;
        const bool ok = cudaPointerGetAttributes(&at, h) == cudaSuccess && at.type == cudaMemoryTypeHost;
        cudaGetLastError();
        return ok;
    };
    if (!(pinned(h_root_state) && pinned(h_actions) && pinned(h_counts) && pinned(h_Q) && pinned(h_V_target) && pinned(h_n_children) &&
          (!h_root_n_init || pinned(h_root_n_init))))
        return fail(AZG_EINVAL, "azg_search_host_begin needs page-locked host buffers (cudaHostAlloc / cudaHostRegister / pin_memory)");
    const size_t cm = e->cmax, Bm = e->cfg.max_trees;
    if (!e->copy_stream) {
        CK(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
        for (int k = 0; k < 2; ++k) {
            CK(cudaEventCreateWithFlags(&e->ev_done[k], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&e->ev_copied[k], cudaEventDisableTiming));
        }
        CK(cudaMallocHost(&e->h_err, 2 * sizeof(int32_t)));
        CK(cudaMalloc(&e->r2_actions, Bm * cm * sizeof(float)));
        CK(cudaMalloc(&e->r2_counts, Bm * cm * sizeof(int32_t)));
        CK(cudaMalloc(&e->r2_Q, Bm * cm * sizeof(double)));
        CK(cudaMalloc(&e->r2_Vt, Bm * sizeof(double)));
        CK(cudaMalloc(&e->r2_nchild, Bm * sizeof(int32_t)));
    }
    float* ra = slot ? e->r2_actions : e->r_actions;
    int32_t* rc_ = slot ? e->r2_counts : e->r_counts;
    double* rq = slot ? e->r2_Q : e->r_Q;
    double* rv = slot ? e->r2_Vt : e->r_Vt;
    int32_t* rn = slot ? e->r2_nchild : e->r_nchild;
    cudaStream_t st = e->own_stream;
    const int sd = state_width(e);
    CK(cudaMemcpyAsync(e->root_state, h_root_state, (size_t)B * sd * sizeof(double), cudaMemcpyHostToDevice, st));
    const int32_t* d_rn = nullptr;
    if (h_root_n_init) {
        CK(cudaMemcpyAsync(e->root_n_init, h_root_n_init, (size_t)B * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        d_rn = e->root_n_init;
    }
    int rc = run_search(e, B, e->root_state, d_rn, n_rollouts, tree_id0, st);
    if (rc) return rc;
    rc = azg_root_results(e, B, ra, rc_, rq, rv, rn, st);
    if (rc) return rc;
    CK(cudaMemcpyAsync(e->h_err + slot, e->err, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CK(cudaMemsetAsync(e->err, 0, sizeof(int32_t), st));
    CK(cudaEventRecord(e->ev_done[slot], st));
    CK(cudaStreamWaitEvent(e->copy_stream, e->ev_done[slot], 0));
    CK(cudaMemcpyAsync(h_actions, ra, (size_t)B * cm * sizeof(float), cudaMemcpyDeviceToHost, e->copy_stream));
    CK(cudaMemcpyAsync(h_counts, rc_, (size_t)B * cm * sizeof(int32_t), cudaMemcpyDeviceToHost, e->copy_stream));
    CK(cudaMemcpyAsync(h_Q, rq, (size_t)B * cm * sizeof(double), cudaMemcpyDeviceToHost, e->copy_stream));
    CK(cudaMemcpyAsync(h_V_target, rv, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, e->copy_stream));
    CK(cudaMemcpyAsync(h_n_children, rn, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost, e->copy_stream));
    CK(cudaEventRecord(e->ev_copied[slot], e->copy_stream));
    e->pending[slot] = true;
    return AZG_OK;
}

extern "C" int azg_search_host_end(azg_engine* e, int32_t slot) {
    if (!e || slot < 0 || slot > 1) return fail(AZG_EINVAL, "bad argument");
    if (!e->pending[slot]) return fail(AZG_EINVAL, "nothing in flight in this slot");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaEventSynchronize(e->ev_copied[slot]));
    e->pending[slot] = false;
    const int32_t h = e->h_err[slot];
    if (h & ERR_NAN) return fail(AZG_ENAN, "NaN in a UCT vector (helpers.py:47-48)");
    if (h & ERR_CAPACITY) return fail(AZG_ECAPACITY, "tree arena or child fan-out capacity exceeded");
    if (h & ERR_WRAP) return fail(AZG_EWRAP, "Acrobot-v1: an angle needed more than 64 iterations of wrap (gym would loop on)");
    return AZG_OK;
}

// host copies of the tree-interleaved tables, back in per-tree order: ctl[t], et[t * 16 + j]
static cudaError_t fetch_ctl(const azg_engine* e, int B, std::vector<CCtl>& out) {
    const size_t BS = e->cfg.max_trees;
    std::vector<uint4> plane(B);
    out.resize(B);
    for (int k = 0; k < 4; ++k) {
        cudaError_t ce = cudaMemcpy(plane.data(), e->ctl + k * BS, (size_t)B * sizeof(uint4), cudaMemcpyDeviceToHost);
        if (ce != cudaSuccess) return ce;
        for (int t = 0; t < B; ++t) reinterpret_cast<uint4*>(&out[t])[k] = plane[t];
    }
    return cudaSuccess;
}
static cudaError_t fetch_et(const azg_engine* e, int B, std::vector<CHot>& out) {
    const size_t BS = e->cfg.max_trees;
    std::vector<CHot> plane(B);
    out.resize((size_t)B * CROOT_MAX_KIDS);
    for (int j = 0; j < CROOT_MAX_KIDS; ++j) {
        cudaError_t ce = cudaMemcpy(plane.data(), e->et + j * BS, (size_t)B * sizeof(CHot), cudaMemcpyDeviceToHost);
        if (ce != cudaSuccess) return ce;
        for (int t = 0; t < B; ++t) out[(size_t)t * CROOT_MAX_KIDS + j] = plane[t];
    }
    return cudaSuccess;
}

extern "C" int azg_get_counters(azg_engine* e, int32_t B, int64_t out[8]) {
    if (!e || !out) return fail(AZG_EINVAL, "null argument");
    if (B < 1 || B > e->cfg.max_trees) return fail(AZG_EINVAL, "B out of range");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaDeviceSynchronize());
    std::vector<uint32_t> c(4 * (size_t)B);
    std::vector<int32_t> dr(B, 0), pw(B, 0);
    // counters are laid out [4][B_of_the_search]; the search that wrote them used last_B
    const int LB = e->last_B > 0 ? e->last_B : B;
    std::vector<uint32_t> all(4 * (size_t)LB);
    CK(cudaMemcpy(all.data(), e->ctr, all.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    if (e->cfg.variant == AZG_DISCRETE) {
        CK(cudaMemcpy(dr.data(), e->draws, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost));
    } else {
        std::vector<CCtl> cc;
        CK(fetch_ctl(e, B, cc));
        for (int t = 0; t < B; ++t) { dr[t] = cc[t].draws; pw[t] = cc[t].pw; }
    }
    for (int k = 0; k < 8; ++k) out[k] = 0;
    const int nb = std::min(B, LB);
    for (int t = 0; t < nb; ++t) {
        out[1] += all[t];
        out[2] += all[(size_t)LB + t];
        out[6] += all[(size_t)2 * LB + t];
        out[4] += all[(size_t)3 * LB + t];
        out[5] += dr[t];
        out[3] += pw[t];
    }
    out[0] = (int64_t)nb * e->last_N;
    out[7] = e->launches;
    return AZG_OK;
}

extern "C" int azg_fused_stats(azg_engine* e, int64_t out[8]) {
    if (!e || !out) return fail(AZG_EINVAL, "null argument");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaDeviceSynchronize());
    unsigned long long h[16];
    CK(cudaMemcpy(h, e->stats, sizeof h, cudaMemcpyDeviceToHost));
    CK(cudaMemset(e->stats, 0, sizeof h));
#ifdef AZG_TREE_PROF
    fprintf(stderr, "tree step sections (cycles summed over warps): load %llu backup %llu select %llu insert %llu expand+store %llu | per-WG total %llu over %llu warpgroups | "
            "discrete level loop: scores %llu draw+pick %llu next row %llu over %llu warp-levels\n", h[8], h[9], h[10], h[11], h[12], h[0], h[4], h[13], h[14], h[11], h[15]);
#endif
#ifdef AZG_EVAL_PROF
    if (e->last_fused_kind == 2)
        fprintf(stderr, "k_search_wg, cycles per warpgroup and search spent waiting for MMAs: at column step 0 of a layer %llu | step 1 %llu | steps 2..7 %llu | kernel %llu\n",
                h[8] / (h[4] ? h[4] : 1), h[9] / (h[4] ? h[4] : 1), h[10] / (h[4] ? h[4] : 1), h[0] / (h[4] ? h[4] : 1));
    else
    fprintf(stderr, "evaluation timeline of epilogue thread 0, cycles per CTA and search: layer 0 %llu | MMA wait %llu | load + convert %llu | stash / quantise / heads %llu | "
            "post-processing wait %llu | tree phase %llu | kernel %llu\n", h[8] / (h[4] ? h[4] : 1), h[9] / (h[4] ? h[4] : 1), h[10] / (h[4] ? h[4] : 1), h[11] / (h[4] ? h[4] : 1),
            h[12] / (h[4] ? h[4] : 1), h[13] / (h[4] ? h[4] : 1), h[0] / (h[4] ? h[4] : 1));
#endif
    for (int k = 0; k < 8; ++k) out[k] = (int64_t)h[k];
    out[5] = e->last_fused_kind;
    return AZG_OK;
}

extern "C" int azg_set_seed(azg_engine* e, uint64_t seed, void* stream) {
    if (!e) return fail(AZG_EINVAL, "null engine");
    CK(cudaSetDevice(e->cfg.device));
    k_set_seed<<<1, 1, 0, (cudaStream_t)stream>>>(e->d_seed, seed);
    CK(cudaGetLastError());
    e->cfg.seed = seed;
    return AZG_OK;
}

extern "C" int azg_set_reward_model(azg_engine* e, double reward_step, double reward_terminal) {
    if (!e) return fail(AZG_EINVAL, "null engine");
    if (!(reward_step == reward_step) || !(reward_terminal == reward_terminal) || std::isinf(reward_step) || std::isinf(reward_terminal))
        return fail(AZG_EINVAL, "rewards must be finite");
    if ((e->cfg.variant != AZG_DISCRETE || e->mc || e->ac) && (reward_step != 1.0 || reward_terminal != 1.0))
        return fail(AZG_EINVAL, "the reward model applies to the CartPole search (the other envs' searches take the env's own reward)");
    if (reward_step == e->reward_step && reward_terminal == e->reward_terminal) return AZG_OK;
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaDeviceSynchronize());
    for (auto& kv : e->graphs) cudaGraphExecDestroy(kv.second);  // captured launches carry the old constants
    e->graphs.clear();
    e->reward_step = reward_step; e->reward_terminal = reward_terminal;
    return AZG_OK;
}

extern "C" uint64_t azg_selfplay_seed(uint64_t seed, int64_t step_index) { return seed + (uint64_t)step_index * 0x9E3779B97F4A7C15ull; }

// One self-play step of B environments: re-key -> search -> root results (the replay row) -> final action -> real env step ->
// episode bookkeeping (selfplay.cuh).  Everything is enqueued on `stream`; nothing synchronises.
extern "C" int azg_selfplay_step(azg_engine* e, int32_t B, const azg_selfplay_io* io, int32_t n_rollouts, int64_t tree_id0,
                                 int64_t step_index, uint64_t base_seed, int32_t max_episode_length, int32_t deterministic,
                                 int32_t by_value, double temperature, void* stream) {
    if (!e || !io) return fail(AZG_EINVAL, "null argument");
    if (!io->d_env_state || !io->d_ep_step || !io->d_episode || !io->d_obs || !io->d_actions || !io->d_counts || !io->d_Q ||
        !io->d_V_target || !io->d_n_children || !io->d_action_taken || !io->d_reward || !io->d_done)
        return fail(AZG_EINVAL, "null buffer in azg_selfplay_io");
    const bool disc = e->cfg.variant == AZG_DISCRETE;
    if (disc && !io->d_root_n) return fail(AZG_EINVAL, "d_root_n is required for the discrete variant");
    if (max_episode_length < 1) return fail(AZG_EINVAL, "max_episode_length must be >= 1");
    if (!(temperature > 0.0)) return fail(AZG_EINVAL, "temperature must be > 0");
    cudaStream_t st = (cudaStream_t)stream;
    int rc = azg_set_seed(e, azg_selfplay_seed(base_seed, step_index), stream);
    if (rc) return rc;
    rc = run_search(e, B, io->d_env_state, disc ? io->d_root_n : nullptr, n_rollouts, tree_id0, st);
    if (rc) return rc;
    rc = azg_root_results(e, B, io->d_actions, io->d_counts, io->d_Q, io->d_V_target, io->d_n_children, stream);
    if (rc) return rc;
    SelfPlayParams sp;
    memset(&sp, 0, sizeof sp);
    sp.B = B; sp.cmax = e->cmax; sp.max_episode_length = max_episode_length; sp.deterministic = deterministic; sp.by_value = by_value;
    sp.temperature = temperature; sp.tree_id0 = tree_id0; sp.seedp = e->d_seed;
    sp.env_state = io->d_env_state; sp.ep_step = io->d_ep_step; sp.episode = io->d_episode; sp.root_n = io->d_root_n;
    sp.actions = io->d_actions; sp.counts = io->d_counts; sp.Q = io->d_Q; sp.n_children = io->d_n_children;
    sp.obs = io->d_obs; sp.action_taken = io->d_action_taken; sp.reward = io->d_reward; sp.done = io->d_done;
    sp.drows = e->drows; sp.R = e->R; sp.err = e->err;
    const int tb = 128, tg = (B + tb - 1) / tb;
    if (disc && e->mc) k_selfplay_discrete<env::MountainCar><<<tg, tb, 0, st>>>(sp);
    else if (disc && e->ac) k_selfplay_discrete<env::Acrobot><<<tg, tb, 0, st>>>(sp);
    else if (disc) k_selfplay_discrete<env::CartPole><<<tg, tb, 0, st>>>(sp);
    else if (e->mcc) k_selfplay_continuous<env::MountainCarContinuous><<<tg, tb, 0, st>>>(sp);
    else k_selfplay_continuous<env::Pendulum><<<tg, tb, 0, st>>>(sp);
    CK(cudaGetLastError());
    return AZG_OK;
}

// ---- tree dump (host side unpacking of the device tables) ------------------------------------------------
// ROW = DRow (CartPole: A = 2, state 4 wide) or D3Row (MountainCar: A = 3, state 2 wide; Acrobot: A = 3, state 4 wide)
template <class ROW>
static int dump_discrete(azg_engine* e, int32_t B, const azg_dump_discrete* o, size_t A, size_t SW) {
    const size_t R = e->R;
    std::vector<ROW> rows((size_t)B * R);
    std::vector<double> st((size_t)B * R * 4);
    std::vector<int32_t> nr(B);
    CK(cudaMemcpy(rows.data(), e->drows, rows.size() * sizeof(ROW), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(st.data(), e->dstate, st.size() * sizeof(double), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(nr.data(), e->n_rows, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost));
    for (size_t t = 0; t < (size_t)B; ++t) {
        o->n_nodes[t] = nr[t];
        for (size_t i = 0; i < R; ++i) {
            const size_t q = t * R + i;
            const bool live = (int)i < nr[t];
            const ROW& r = rows[q];
            o->parent[q] = live ? (r.parent == DROW_NONE ? -1 : r.parent) : 0;
            o->paction[q] = live ? (r.parent == DROW_NONE ? -1 : r.paction) : 0;
            o->node_n[q] = live ? r.node_n : 0;
            o->terminal[q] = live ? (r.flags & ROW_TERMINAL) : 0;
            o->V[q] = live ? r.V : 0.0f;
            o->r[q] = live ? r.r : 0.0;
            for (size_t k = 0; k < SW; ++k) o->state[q * SW + k] = live ? st[q * 4 + k] : 0.0;
            for (size_t a = 0; a < A; ++a) {
                o->prior[q * A + a] = live ? r.prior[a] : 0.0f;
                o->eW[q * A + a] = live ? r.W[a] : 0.0;
                o->en[q * A + a] = live ? r.n_e[a] : 0;
                o->echild[q * A + a] = live ? (r.child[a] == DROW_NONE ? -1 : r.child[a]) : 0;
            }
        }
    }
    return AZG_OK;
}

extern "C" int azg_dump_tree_discrete(azg_engine* e, int32_t B, const azg_dump_discrete* o) {
    if (!e || !o) return fail(AZG_EINVAL, "null argument");
    if (e->cfg.variant != AZG_DISCRETE) return fail(AZG_EINVAL, "engine is not discrete");
    if (B < 1 || B > e->cfg.max_trees) return fail(AZG_EINVAL, "B out of range");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaDeviceSynchronize());
    if (e->mc) return dump_discrete<D3Row>(e, B, o, 3, 2);
    if (e->ac) return dump_discrete<D3Row>(e, B, o, 3, 4);
    return dump_discrete<DRow>(e, B, o, 2, 4);
}

extern "C" int azg_dump_tree_continuous(azg_engine* e, int32_t B, const azg_dump_continuous* o) {
    if (!e || !o) return fail(AZG_EINVAL, "null argument");
    if (e->cfg.variant != AZG_CONTINUOUS) return fail(AZG_EINVAL, "engine is not continuous");
    if (B < 1 || B > e->cfg.max_trees) return fail(AZG_EINVAL, "B out of range");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaDeviceSynchronize());
    const size_t R = e->R, K3 = e->K3, HS = e->HS;
    std::vector<CRow> rows((size_t)B * R);
    std::vector<CHot> et;
    std::vector<CCtl> ctl;
    std::vector<float> hd((size_t)B * R * HS);
    CK(cudaMemcpy(rows.data(), e->crows, rows.size() * sizeof(CRow), cudaMemcpyDeviceToHost));
    CK(fetch_et(e, B, et));
    CK(fetch_ctl(e, B, ctl));
    CK(cudaMemcpy(hd.data(), e->chead, hd.size() * sizeof(float), cudaMemcpyDeviceToHost));
    std::vector<int32_t> par(R);
    std::vector<const CHot*> hot(R);
    for (size_t t = 0; t < (size_t)B; ++t) {
        const int nr = ctl[t].n_rows;
        o->n_rows[t] = nr;
        // parent links are implicit in the child lists; root children keep their statistics in the edge table
        for (size_t i = 0; i < R; ++i) { par[i] = -1; hot[i] = reinterpret_cast<const CHot*>(&rows[t * R + i]); }
        for (int k = 0; k < ctl[t].root_nk && k < CROOT_MAX_KIDS; ++k) {
            const size_t kid = ctl[t].root_kids[k];
            if (kid < R) { par[kid] = 0; hot[kid] = &et[t * CROOT_MAX_KIDS + k]; }
        }
        for (size_t i = 1; i < R && (int)i < nr; ++i) {
            if (!(hot[i]->nn_flags & CROW_EXPANDED)) continue;
            const CRow& r = rows[t * R + i];
            for (int k = 0; k < r.nkids && k < CROW_MAX_KIDS; ++k)
                if (r.kids[k] < R) par[r.kids[k]] = (int32_t)i;
        }
        for (size_t i = 0; i < R; ++i) {
            const size_t q = t * R + i;
            const bool live = (int)i < nr;
            const CHot& h = *hot[i];
            const CRow& r = rows[q];
            const bool ex = live && (h.nn_flags & CROW_EXPANDED);
            o->parent[q] = live ? par[i] : 0;
            o->action[q] = live && i > 0 ? h.action : 0.0f;
            o->eW[q] = live ? h.W : 0.0;
            o->en[q] = live ? h.n_e : 0;
            o->expanded[q] = ex ? 1 : 0;
            o->node_n[q] = ex ? (i == 0 ? ctl[t].root_nn : (int32_t)(h.nn_flags & CROW_NMASK)) : 0;
            o->terminal[q] = ex && (h.nn_flags & CROW_TERMINAL) ? 1 : 0;
            o->V[q] = ex ? h.V : 0.0f;
            o->r[q] = ex ? h.r : 0.0;
            o->state[q * 2] = ex ? r.th : 0.0;
            o->state[q * 2 + 1] = ex ? r.thdot : 0.0;
            for (size_t k = 0; k < K3; ++k) o->head[q * K3 + k] = ex ? hd[q * HS + k] : 0.0f;
        }
    }
    return AZG_OK;
}

// ---- standalone building blocks for known-answer tests --------------------------------------------------
extern "C" int azg_mlp_forward(azg_engine* e, int32_t n, const float* d_x, float* d_V, float* d_head, void* stream) {
    if (!e || !d_x || !d_V || !d_head) return fail(AZG_EINVAL, "null argument");
    if (n < 1) return fail(AZG_EINVAL, "n must be >= 1");
    if (!e->weights_set) return fail(AZG_EINVAL, "azg_set_weights has not been called");
    CK(cudaSetDevice(e->cfg.device));
    MlpParams m = make_mlp_params(e, n);
    m.X = d_x; m.xstride = e->cfg.state_dim; m.mode = 1; m.outV = d_V; m.outHead = d_head; m.evals = nullptr;
    CK(launch_mlp(e, m, (cudaStream_t)stream, false));
    return AZG_OK;
}

template <class ENV>
__device__ __forceinline__ void env_step_continuous(int i, const double* s, const float* a, double* o, double* rew, int32_t* term, float* obs) {
    double n0, n1, r;
    const bool t = ENV::step(s[i * 2], s[i * 2 + 1], a[i], n0, n1, r);
    o[i * 2] = n0; o[i * 2 + 1] = n1;
    const float4 ob = ENV::obs(n0, n1);
    obs[i * ENV::S] = ob.x; obs[i * ENV::S + 1] = ob.y;
    if (ENV::S > 2) obs[i * ENV::S + 2] = ob.z;
    rew[i] = r;
    term[i] = t;
}

__global__ void k_env_step(int variant, bool mcc, bool mc, bool ac, int n, const double* s, const float* a, double* o, double* rew,
                           int32_t* term, float* obs, int32_t* err) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (variant == AZG_DISCRETE && ac) {  // the action is an index 0, 1, 2; the observation is 6 wide
        const double in[4] = {s[i * 4], s[i * 4 + 1], s[i * 4 + 2], s[i * 4 + 3]};
        double out[4], r;
        bool capped = false;
        const bool t = env::acrobot_step(in, (int)a[i], out, r, capped);
        if (capped) atomicOr(err, ERR_WRAP);
        float x[6];
        env::acrobot_obs(out, x);
        for (int k = 0; k < 4; ++k) o[i * 4 + k] = out[k];
        for (int k = 0; k < 6; ++k) obs[i * 6 + k] = x[k];
        rew[i] = r;
        term[i] = t;
    } else if (variant == AZG_DISCRETE && mc) {  // the action is an index 0, 1, 2
        double n0, n1, r;
        const bool t = env::MountainCar::step(s[i * 2], s[i * 2 + 1], (int)a[i], n0, n1, r);
        o[i * 2] = n0; o[i * 2 + 1] = n1;
        obs[i * 2] = (float)n0; obs[i * 2 + 1] = (float)n1;
        rew[i] = r;
        term[i] = t;
    } else if (variant == AZG_DISCRETE) {
        const double in[4] = {s[i * 4], s[i * 4 + 1], s[i * 4 + 2], s[i * 4 + 3]};
        double out[4], r;
        const bool t = env::cartpole_step(in, (int)a[i], out, r);
        for (int k = 0; k < 4; ++k) { o[i * 4 + k] = out[k]; obs[i * 4 + k] = (float)out[k]; }
        rew[i] = r;
        term[i] = t;
    } else if (mcc) {
        env_step_continuous<env::MountainCarContinuous>(i, s, a, o, rew, term, obs);
    } else {
        env_step_continuous<env::Pendulum>(i, s, a, o, rew, term, obs);
    }
}

extern "C" int azg_env_step(azg_engine* e, int32_t n, const double* d_state, const float* d_action, double* d_next, double* d_reward,
                            int32_t* d_terminal, float* d_obs, void* stream) {
    if (!e || !d_state || !d_action || !d_next || !d_reward || !d_terminal || !d_obs) return fail(AZG_EINVAL, "null argument");
    if (n < 1) return fail(AZG_EINVAL, "n must be >= 1");
    CK(cudaSetDevice(e->cfg.device));
    k_env_step<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(e->cfg.variant, e->mcc, e->mc, e->ac, n, d_state, d_action, d_next, d_reward,
                                                                  d_terminal, d_obs, e->err);
    CK(cudaGetLastError());
    return AZG_OK;
}

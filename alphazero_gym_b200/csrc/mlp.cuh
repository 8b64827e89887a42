// mlp.cuh -- batched leaf evaluation: trunk MLP + value head + policy head in ONE kernel.
//
// Replaces the batch-1 model.predict_V / predict_pi / sample_action calls the reference makes per node
// (mcts.py:406-416, :619-623, :652 -> policies.py:154-160, :340-352, :656-669).  The trunk runs once per
// leaf (the reference runs it 2x per discrete node and again for every progressive-widening sample) and
// the post-processed policy head is cached with the node.
//
// Arithmetic: FP32 FMA, NOT tensor cores.  BASELINE.json's tolerance (Q/V within 1e-5, bit-exact visit
// counts) rules out TF32/BF16 products, and a fixed summation order -- acc = bias; acc = fma(w[j][k],
// x[k], acc) for k ascending -- makes every output bit-reproducible by the CPU oracle.  A register-tiled
// SGEMM has exactly that per-output order as long as k is the outer loop.
//
// Structure (one persistent CTA per SM, 512 threads for H = 128):
//   * all weights (138 KB for 3x128 ELU, 71 KB for 2x128 ReLU) are staged in shared memory once per CTA
//     with TMA bulk copies (cp.async.bulk + mbarrier) and reused for every unit the CTA processes;
//   * rows are dealt to CTAs in units of 32 (65536 rows = 2048 units = 13.8 per SM, so the tail is 1.2 %);
//   * activations live in shared memory k-major ([H][32] per group); both operands of the register tile
//     are read with conflict-free LDS.128 and the K loop is software-pipelined (operands of k+1 are in
//     flight while the FMAs of k issue);
//   * activations are branch-free (ELU through the deterministic expm1 of detmath.cuh).
// Bound: FP32 FMA issue (2*H*H flop per row per hidden layer).
#pragma once
#include "common.cuh"
#include "detmath.cuh"

#define MLP_MAX_PO 28  // 1 + 3*AZG_MAX_K rounded up to a multiple of 4

struct MlpParams {
    const float* wpack;  // packed weights (engine.cu pack_weights): per layer Wt[K][H] k-major + b[H]; heads Wh[H][PO_PAD] + bh[PO_PAD]
    int32_t wcount;      // floats in wpack (multiple of 4)
    int32_t L, P, PO_PAD;
    int32_t n;           // rows to evaluate
    const float* X;      // [n][xstride]
    int32_t xstride;
    int32_t mode;        // 0: scatter into the tree tables of leaf[] rows; 1: dense outputs
    int32_t variant, A, K, R, HS;
    float ls_min, ls_max;
    const int32_t* leaf;
    DRow* drows;
    CRow* crows;
    float* chead;
    uint32_t* evals;     // per-tree evaluation counter
    uint4* ctl;          // continuous: control-block chunk planes [4][BS] (common.cuh): leaf word; leafR += gamma_f32 * V (mcts.py:260-263)
    CHot* et;            // continuous: root edge table [16][BS] (V of a root child is written there)
    int32_t BS;          // plane stride of the tree-interleaved tables (max_trees)
    float gamma_f32;
    float* outV;
    float* outHead;
    int32_t head_dim;
    // AZG_FLAG_EVAL_Q8 (qmlp.cuh): int8 digit planes [L-1][3][H/16][H][16] and the f32 side table (engine.cu pack_weights_q8)
    const int8_t* qdigits;
    const int8_t* qdigits_nat;  // the same digit planes with the rows in natural order (search_wg.cuh)
    const float* qfl;
    int32_t qfl_count;  // floats in qfl (multiple of 4)
    // whole-search kernel: cycle accounting, summed over CTAs (azg_fused_stats, include/azg.h)
    unsigned long long* stats;
};

// ---- TMA bulk copy global -> shared, completion on an mbarrier (SASS: UBLKCP / SYNCS) --------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// the same with a suspend-time hint (ns): the warp sleeps inside the instruction until the phase completes or the time is up,
// instead of coming back every few hundred cycles to spin (a quarter of all issued instructions of the first whole-search kernel
// were wait loops, profiles/r1f)
__device__ __forceinline__ bool mbar_try_wait_hint(uint64_t* bar, uint32_t parity, uint32_t ns) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity), "r"(ns)
        : "memory");
    return ok != 0;
}

// ---- activations (branch-free) -------------------------------------------------------------------------
// rint(t) and 2^rint(t) without the conversion (XU) pipe, for t in [-2^22, 2^22]: adding 1.5 * 2^23 rounds t to the nearest-even
// integer (the IEEE addition does the rounding) and leaves that integer in the low mantissa bits.  Same values as rintf / the
// f32 -> s32 conversion, but FADD + integer ops instead of FRND + F2I, which run at a quarter of the FMA rate and bounded the
// evaluation kernels (profiles/r1c: XU pipe 78 % busy).
#define MLP_RINT_MAGIC 12582912.0f
__device__ __forceinline__ float mlp_pow2_of_magic(float tm) {  // tm = t + MAGIC  ->  2^rint(t)
    return __uint_as_float((__float_as_uint(tm) << 23) + 0x3F800000u);
}

// the activations of the reference's map beyond ReLU / ELU (alphazero/network/utils.py:5-14), each the scalar f32 operation
// sequence of the torch CPU kernel it replaces; SiLU through the deterministic expf (<= 1 ulp from torch's)
__device__ __forceinline__ float mlp_act_other(int act, float v) {
    if (act == 2) return v > 0.0f ? v : __fmul_rn(v, 0.01f);                                     // LeakyReLU(0.01)
    if (act == 3) return fminf(fmaxf(v, 0.0f), 6.0f);                                             // ReLU6
    if (act == 4) return (v != v) ? v : __fdiv_rn(v, __fadd_rn(1.0f, det::expf_(-v)));            // SiLU: x / (1 + exp(-x))
    return __fdiv_rn(__fmul_rn(v, fminf(fmaxf(__fadd_rn(v, 3.0f), 0.0f), 6.0f)), 6.0f);           // Hardswish: x * relu6(x + 3) / 6
}

template <int ACT>
__device__ __forceinline__ float mlp_act(float v) {
    if (ACT >= 2) return mlp_act_other(ACT, v);
    if (ACT == 0) return v > 0.0f ? v : 0.0f;  // ReLU (DiscretePolicy.yaml:8)
    // ELU alpha=1 (ContinuousPolicy.yaml:9): v > 0 ? v : expm1(v), expm1 = det::expm1f_ written with selects.
    // (n == 0 needs no special case: fma(p, 1, 0) == p; for v > 0 the exponential branch is computed on garbage and discarded.)
    const float xx = fmaxf(v, -20.0f);
    const float tm = __fadd_rn(__fmul_rn(xx, 1.44269504088896341f), MLP_RINT_MAGIC);
    const float n = __fsub_rn(tm, MLP_RINT_MAGIC);
    float r = __fmaf_rn(n, -0.693359375f, xx);
    r = __fmaf_rn(n, 2.12194440e-4f, r);
    const float pl = det::expm1_poly(r);
    const float t = mlp_pow2_of_magic(tm);
    const float e = __fmaf_rn(pl, t, __fsub_rn(t, 1.0f));
    // Two selects of the reference form are redundant here and dropped (same bits, two FSETP + two FSEL fewer per element on the
    // evaluation kernels' critical pipe): for EVERY f32 v < -17.5 the clamped evaluation already yields exactly -1.0f (t <= 2^-25,
    // so t - 1 and the final fma round to -1; checked exhaustively over all 1 039 400 960 such values, tools/elu_check.c), and
    // "v <= 0 ? e : v" passes a NaN through by itself.
    return v <= 0.0f ? e : v;
}

// the same activation on a pair, with the FMA-pipe work packed into f32x2 instructions (each half is the scalar
// IEEE operation, so results are bit-identical to mlp_act on each element)
template <int ACT>
__device__ __forceinline__ float2 mlp_act2(float2 v) {
    if (ACT >= 2) return make_float2(mlp_act_other(ACT, v.x), mlp_act_other(ACT, v.y));
    if (ACT == 0) return make_float2(v.x > 0.0f ? v.x : 0.0f, v.y > 0.0f ? v.y : 0.0f);
    const float2 xx = make_float2(fmaxf(v.x, -20.0f), fmaxf(v.y, -20.0f));
    const float2 magic = make_float2(MLP_RINT_MAGIC, MLP_RINT_MAGIC);
    const float2 tm = __fadd2_rn(__fmul2_rn(xx, make_float2(1.44269504088896341f, 1.44269504088896341f)), magic);
    const float2 n = __fadd2_rn(tm, make_float2(-MLP_RINT_MAGIC, -MLP_RINT_MAGIC));
    float2 r = __ffma2_rn(n, make_float2(-0.693359375f, -0.693359375f), xx);
    r = __ffma2_rn(n, make_float2(2.12194440e-4f, 2.12194440e-4f), r);
    float2 p = make_float2(1.9875691500E-4f, 1.9875691500E-4f);
    p = __ffma2_rn(p, r, make_float2(1.3981999507E-3f, 1.3981999507E-3f));
    p = __ffma2_rn(p, r, make_float2(8.3334519073E-3f, 8.3334519073E-3f));
    p = __ffma2_rn(p, r, make_float2(4.1665795894E-2f, 4.1665795894E-2f));
    p = __ffma2_rn(p, r, make_float2(1.6666665459E-1f, 1.6666665459E-1f));
    p = __ffma2_rn(p, r, make_float2(5.0000001201E-1f, 5.0000001201E-1f));
    const float2 z = __fmul2_rn(r, r);
    const float2 pl = __ffma2_rn(p, z, r);
    const float2 t = make_float2(mlp_pow2_of_magic(tm.x), mlp_pow2_of_magic(tm.y));
    const float2 e = __ffma2_rn(pl, t, __fadd2_rn(t, make_float2(-1.0f, -1.0f)));
    return make_float2(v.x <= 0.0f ? e.x : v.x, v.y <= 0.0f ? e.y : v.y);  // see mlp_act: the saturation and NaN selects are redundant
}

// post-processing of one row's raw head outputs (policies.py:275-297 softmax priors; :617-631 GMM params)
__device__ __forceinline__ void softmax_seq(const float* l, int n, float* p) {
    float m = l[0];
    for (int i = 1; i < n; ++i) m = l[i] > m ? l[i] : m;
    float s = 0.0f;
    for (int i = 0; i < n; ++i) {
        p[i] = det::expf_(__fsub_rn(l[i], m));
        s = __fadd_rn(s, p[i]);
    }
    for (int i = 0; i < n; ++i) p[i] = __fdiv_rn(p[i], s);
}

// mode 0, continuous tree, compile-time K: the same values as the generic path below with every array index static, so that raw[] and
// post[] live in registers (the run-time-K version goes through local memory; in the whole-search kernel, which has almost no L1, that
// was 2.3 us per simulation the evaluation warps spent waiting for the post-processing warps at the phase boundary)
template <int K>
__device__ __forceinline__ void finish_row_continuous(const MlpParams& p, int gr, int leafw, double lr, float V, const float* raw) {
    constexpr int NP = 3 * K, HSK = (NP + 3) / 4 * 4;
    float post[HSK];
#pragma unroll
    for (int i = 0; i < HSK; ++i) post[i] = 0.0f;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        post[k] = raw[k];
        float ls = raw[K + k];
        ls = ls < p.ls_min ? p.ls_min : ls;
        ls = ls > p.ls_max ? p.ls_max : ls;
        post[K + k] = det::expf_(ls);
    }
    if (K > 1) {  // softmax_seq over the K mixture logits, same operation order
        float m = raw[2 * K];
#pragma unroll
        for (int i = 1; i < K; ++i) m = raw[2 * K + i] > m ? raw[2 * K + i] : m;
        float sum = 0.0f;
#pragma unroll
        for (int i = 0; i < K; ++i) {
            post[2 * K + i] = det::expf_(__fsub_rn(raw[2 * K + i], m));
            sum = __fadd_rn(sum, post[2 * K + i]);
        }
#pragma unroll
        for (int i = 0; i < K; ++i) post[2 * K + i] = __fdiv_rn(post[2 * K + i], sum);
    } else {
        post[2] = 1.0f;
    }
    const size_t ri = (size_t)gr * p.R + (leafw & LEAF_ROW_MASK);
    if (leafw & LEAF_TERMINAL) V = 0.0f;  // mcts.py:619-623
    if (leafw & LEAF_ROOTCHILD) p.et[(size_t)((leafw >> LEAF_J_SHIFT) & 0xFF) * p.BS + gr].V = V;
    else p.crows[ri].V = V;
    reinterpret_cast<double*>(p.ctl + (size_t)p.BS + gr)[1] = lr + (double)__fmul_rn(p.gamma_f32, V);  // CCtl::leafR = chunk 1, bytes 8..15
    float4* h = reinterpret_cast<float4*>(p.chead + ri * p.HS);
#pragma unroll
    for (int i = 0; i < HSK / 4; ++i) h[i] = make_float4(post[4 * i], post[4 * i + 1], post[4 * i + 2], post[4 * i + 3]);
}

// post-processing + write-back of one evaluated row: V and the raw policy-head outputs -> softmax priors / GMM parameters ->
// the tree tables (mode 0) or dense outputs (mode 1).  Shared by k_mlp, k_qmlp2 and k_search_wg; the caller counts the evaluation.
// ROW3: the discrete tree may hold three-action rows (D3Row, MountainCar-v0), told apart by p.A at run time.  k_mlp serves every env
// and passes true; the k_qmlp2 / k_search_wg instantiations know their env and pass whether it is MountainCar.
template <bool ROW3>
__device__ __forceinline__ void mlp_finish_row(const MlpParams& p, int gr, int leafw, double lr, float V, const float* raw) {
    if (p.mode == 0 && p.variant == 0 && p.A == 2) {  // CartPole: softmax_seq over two logits, written out (registers only)
        const float m = raw[1] > raw[0] ? raw[1] : raw[0];
        const float e0 = det::expf_(__fsub_rn(raw[0], m)), e1 = det::expf_(__fsub_rn(raw[1], m));
        const float sum = __fadd_rn(__fadd_rn(0.0f, e0), e1);
        DRow* d = p.drows + (size_t)gr * p.R + (leafw & LEAF_ROW_MASK);
        d->V = (leafw & LEAF_TERMINAL) ? 0.0f : V;  // mcts.py:406-410
        *reinterpret_cast<float2*>(d->prior) = make_float2(__fdiv_rn(e0, sum), __fdiv_rn(e1, sum));
        return;
    }
    if constexpr (ROW3) {
        if (p.mode == 0 && p.variant == 0 && p.A == 3) {  // MountainCar: softmax_seq over three logits into line 0 of the D3Row
            float pr[3];
            softmax_seq(raw, 3, pr);
            D3Row* d = reinterpret_cast<D3Row*>(p.drows) + (size_t)gr * p.R + (leafw & LEAF_ROW_MASK);
            d->V = (leafw & LEAF_TERMINAL) ? 0.0f : V;
            d->prior[0] = pr[0]; d->prior[1] = pr[1]; d->prior[2] = pr[2];
            return;
        }
    }
    if (p.mode == 0 && p.variant == 1) {
        switch (p.K) {
            case 1: finish_row_continuous<1>(p, gr, leafw, lr, V, raw); return;
            case 2: finish_row_continuous<2>(p, gr, leafw, lr, V, raw); return;
            case 3: finish_row_continuous<3>(p, gr, leafw, lr, V, raw); return;
            case 4: finish_row_continuous<4>(p, gr, leafw, lr, V, raw); return;
            default: break;
        }
    }
    float post[3 * AZG_MAX_K];
    int npost;
    if (p.variant == 0) {
        softmax_seq(raw, p.A, post);
        npost = p.A;
    } else {
        const int K = p.K;
        for (int k = 0; k < K; ++k) {
            post[k] = raw[k];
            float ls = raw[K + k];
            ls = ls < p.ls_min ? p.ls_min : ls;
            ls = ls > p.ls_max ? p.ls_max : ls;
            post[K + k] = det::expf_(ls);
        }
        if (K > 1) softmax_seq(raw + 2 * K, K, post + 2 * K);
        else post[2] = 1.0f;
        npost = 3 * K;
    }
    if (p.mode == 1) {
        p.outV[gr] = V;
        for (int i = 0; i < npost; ++i) p.outHead[(size_t)gr * p.head_dim + i] = post[i];
    } else {
        const size_t ri = (size_t)gr * p.R + (leafw & LEAF_ROW_MASK);
        if (leafw & LEAF_TERMINAL) V = 0.0f;  // mcts.py:406-410, :619-623
        if (p.variant == 0) {
            DRow* d = p.drows + ri;
            d->V = V;
            *reinterpret_cast<float2*>(d->prior) = make_float2(post[0], post[1]);
        } else {
            if (leafw & LEAF_ROOTCHILD) p.et[(size_t)((leafw >> LEAF_J_SHIFT) & 0xFF) * p.BS + gr].V = V;
            else p.crows[ri].V = V;
            reinterpret_cast<double*>(p.ctl + (size_t)p.BS + gr)[1] = lr + (double)__fmul_rn(p.gamma_f32, V);  // CCtl::leafR = chunk 1, bytes 8..15
            float* h = p.chead + ri * p.HS;  // HS is a multiple of 4 floats: vector stores
            for (int i = 0; i < npost; i += 4)
                *reinterpret_cast<float4*>(h + i) = make_float4(post[i], i + 1 < npost ? post[i + 1] : 0.0f, i + 2 < npost ? post[i + 2] : 0.0f,
                                                                i + 3 < npost ? post[i + 3] : 0.0f);
        }
    }
}

// Thread mapping.  The CTA (512 threads for H = 128) is split into NGRP = 4 independent groups of H/32
// warps.  A group owns a unit of 32 rows at a time: its private [H][32] activation buffer, its own named
// barrier (bar.sync id, 128) -- never a CTA-wide __syncthreads in the steady state.  All groups share the
// weights staged once in shared memory.  Because groups are decoupled they drift out of phase, so one
// group's activation / head / write-back instructions fill the issue slots another group's FMA loop
// leaves free (the lock-step 16-warp version stalled on math-pipe throttle and barriers together,
// profiles/r1c).  Inside a group each warp owns 32 rows x 32 columns, each thread 4 rows x 8 columns; per k
// a warp reads 128 B of activations (LDS.128, 8 distinct lanes, rest broadcast) and 2 x 64 B of weights.
// The accumulators are float2 column pairs updated with the packed fma.rn.f32x2 (SASS FFMA2, scalar operand
// broadcast): half the issue slots of scalar FFMA for the same IEEE result per element.  k is the outer
// loop, so every output still sums in k order.
#define MLP_NGRP 4
#define MLP_UNIT 32
#define MLP_GTHREADS(H) (32 * ((H) / 32))
#define MLP_THREADS(H) (MLP_NGRP * MLP_GTHREADS(H))

__device__ __forceinline__ void group_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

template <int H, int ACT>
__device__ __forceinline__ void hidden_layer(const float* __restrict__ Wt, const float* __restrict__ b, float* actg, int gt, int bar) {
    constexpr int TU = MLP_UNIT;
    const int lane = gt & 31, wc = gt >> 5;  // warp column block (32 cols)
    const int row0 = (lane & 7) * 4, col0 = wc * 32 + (lane >> 3) * 8;
#ifndef MLP_UNROLL
#define MLP_UNROLL 16
#endif
#define MLP_STR2(x) #x
#define MLP_STR(x) MLP_STR2(x)
    const float* ap = actg + row0;
    const float* wp = Wt + col0;
    float4 a = *reinterpret_cast<const float4*>(ap);
    float4 w0 = *reinterpret_cast<const float4*>(wp);
    float4 w1 = *reinterpret_cast<const float4*>(wp + 4);
    // accumulators paired along columns: acc[r][c] = (column 2c, column 2c+1) of row r; the activation is the scalar operand
    float2 acc[4][4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const float2 bc = *reinterpret_cast<const float2*>(b + col0 + 2 * c);
#pragma unroll
        for (int r = 0; r < 4; ++r) acc[r][c] = bc;
    }
    _Pragma(MLP_STR(unroll MLP_UNROLL))
    for (int k = 0; k < H; ++k) {
        const int kn = k + 1 < H ? k + 1 : k;  // the last iteration re-reads row k (discarded)
        const float4 na = *reinterpret_cast<const float4*>(ap + kn * TU);
        const float4 nw0 = *reinterpret_cast<const float4*>(wp + kn * H);
        const float4 nw1 = *reinterpret_cast<const float4*>(wp + kn * H + 4);
        const float ar[4] = {a.x, a.y, a.z, a.w};
        const float2 wpair[4] = {make_float2(w0.x, w0.y), make_float2(w0.z, w0.w), make_float2(w1.x, w1.y), make_float2(w1.z, w1.w)};
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const float2 av = make_float2(ar[r], ar[r]);
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[r][c] = __ffma2_rn(av, wpair[c], acc[r][c]);
        }
        a = na; w0 = nw0; w1 = nw1;
    }
    group_sync(bar, MLP_GTHREADS(H));  // the whole group has finished reading this layer's input
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        float* d0 = actg + (col0 + 2 * c) * TU + row0;
        const float2 e0 = mlp_act2<ACT>(acc[0][c]), e1 = mlp_act2<ACT>(acc[1][c]), e2 = mlp_act2<ACT>(acc[2][c]), e3 = mlp_act2<ACT>(acc[3][c]);
        *reinterpret_cast<float4*>(d0) = make_float4(e0.x, e1.x, e2.x, e3.x);
        *reinterpret_cast<float4*>(d0 + TU) = make_float4(e0.y, e1.y, e2.y, e3.y);
    }
    group_sync(bar, MLP_GTHREADS(H));
}

// one unit of 32 rows, executed by one group of H/32 warps
template <int H, int S, int ACT>
__device__ __forceinline__ void mlp_unit(const MlpParams& p, const float* w, float* actg, float* outg, int row0, int gt, int bar) {
    constexpr int TU = MLP_UNIT;
    constexpr int NQ = MLP_GTHREADS(H) / TU;  // threads per row in the row-per-thread phases (H=128: 4)
    const int row = gt % TU, q = gt / TU;
    const int gr = row0 + row;
    int leafw = 0;
    bool need = gr < p.n;
    double lr = 0.0;
    if (need && p.mode == 0) {
        if (p.variant == 1) {  // continuous: leaf word and leafR share the first 32 B of the control block
            const uint4 c0 = p.ctl[gr], c1 = p.ctl[(size_t)p.BS + gr];
            leafw = (int)c0.z;
            lr = __hiloint2double((int)c1.w, (int)c1.z);
        } else {
            leafw = p.leaf[gr];
        }
        need = (leafw & LEAF_EVAL) != 0;
    }
    // ---- layer 0: S -> H, NQ threads per row, H/NQ outputs each
    {
        float x[S];
#pragma unroll
        for (int s = 0; s < S; ++s) x[s] = 0.0f;
        if (need) {
            if (p.xstride == 4) {
                const float4 v = *reinterpret_cast<const float4*>(p.X + (size_t)gr * 4);
                x[0] = v.x; x[1] = v.y;
                if constexpr (S > 2) x[2] = v.z;
                if (S > 3) x[S - 1] = v.w;
            } else {
#pragma unroll
                for (int s = 0; s < S; ++s) x[s] = p.X[(size_t)gr * p.xstride + s];
            }
        }
        const float* W0 = w;
        const float* b0 = w + S * H;
#pragma unroll 4
        for (int j = q * (H / NQ); j < (q + 1) * (H / NQ); j += 2) {
            float2 acc = *reinterpret_cast<const float2*>(b0 + j);
#pragma unroll
            for (int s = 0; s < S; ++s)
                acc = __ffma2_rn(make_float2(x[s], x[s]), *reinterpret_cast<const float2*>(W0 + s * H + j), acc);
            const float2 e = mlp_act2<ACT>(acc);
            actg[j * TU + row] = e.x;
            actg[(j + 1) * TU + row] = e.y;
        }
    }
    group_sync(bar, MLP_GTHREADS(H));
    // ---- hidden layers
    int off = S * H + H;
    for (int l = 1; l < p.L; ++l) {
        hidden_layer<H, ACT>(w + off, w + off + H * H, actg, gt, bar);
        off += H * H + H;
    }
    // ---- heads: column 0 = value_head, columns 1..P = dist_head; 4 outputs per thread and pass
    {
        const float* Wh = w + off;
        const float* bh = Wh + H * p.PO_PAD;
        for (int c = q; c < p.PO_PAD / 4; c += NQ) {
            const float4 b4 = *reinterpret_cast<const float4*>(bh + c * 4);
            float2 lo = make_float2(b4.x, b4.y), hi = make_float2(b4.z, b4.w);
#pragma unroll 8
            for (int k = 0; k < H; ++k) {
                const float a = actg[k * TU + row];
                const float4 w4 = *reinterpret_cast<const float4*>(Wh + k * p.PO_PAD + c * 4);
                const float2 av = make_float2(a, a);
                lo = __ffma2_rn(av, make_float2(w4.x, w4.y), lo);
                hi = __ffma2_rn(av, make_float2(w4.z, w4.w), hi);
            }
            const float4 acc = make_float4(lo.x, lo.y, hi.x, hi.y);
            outg[(c * 4 + 0) * TU + row] = acc.x;
            outg[(c * 4 + 1) * TU + row] = acc.y;
            outg[(c * 4 + 2) * TU + row] = acc.z;
            outg[(c * 4 + 3) * TU + row] = acc.w;
        }
    }
    group_sync(bar, MLP_GTHREADS(H));
    // ---- post-processing + write-back: one thread per row (warp 0 of the group); the group's other warps run
    // ahead into the next unit's layer 0 (they only touch actg, and outg is not rewritten before two more
    // group barriers that warp 0 takes part in)
    if (q == 0 && need) {
        float raw[3 * AZG_MAX_K];
        for (int i = 0; i < p.P; ++i) raw[i] = outg[(1 + i) * TU + row];
        mlp_finish_row<true>(p, gr, leafw, lr, outg[row], raw);  // k_mlp serves every env: the row layout is known at run time
        if (p.mode == 0) p.evals[gr] += 1;
    }
}

template <int H, int S, int ACT>
__global__ void __launch_bounds__(MLP_THREADS(H), 1) k_mlp(const MlpParams p) {
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) uint64_t wbar;
    const int tid = threadIdx.x;
    const int grp = tid / MLP_GTHREADS(H), gt = tid % MLP_GTHREADS(H);
    float* w = smem;
    float* actg = smem + p.wcount + grp * (H + p.PO_PAD) * MLP_UNIT;  // [H][32] activations of this group
    float* outg = actg + H * MLP_UNIT;                               // [PO_PAD][32] raw head outputs

    // rows are dealt in units of 32: CTA b owns units [b*per, (b+1)*per), group g takes every 4th of them
    const int units = (p.n + MLP_UNIT - 1) / MLP_UNIT;
    const int per = (units + gridDim.x - 1) / gridDim.x;
    const int unit0 = blockIdx.x * per;
    const int unit_end = min(unit0 + per, units);
    if (unit0 >= unit_end) return;

    // stage all weights with TMA bulk copies; every thread then waits on the mbarrier
    if (tid == 0) mbar_init(&wbar, 1);
    __syncthreads();
    if (tid == 0) {
        const uint32_t bytes = (uint32_t)p.wcount * 4u;
        mbar_expect_tx(&wbar, bytes);
        for (uint32_t o = 0; o < bytes; o += 32768u)
            bulk_g2s(reinterpret_cast<char*>(w) + o, reinterpret_cast<const char*>(p.wpack) + o, min(32768u, bytes - o), &wbar);
    }
    while (!mbar_try_wait(&wbar, 0)) {}

    for (int unit = unit0 + grp; unit < unit_end; unit += MLP_NGRP)
        mlp_unit<H, S, ACT>(p, w, actg, outg, unit * MLP_UNIT, gt, 1 + grp);
}

// qmlp2.cuh -- batched leaf evaluation on the 5th-generation tensor cores, two row tiles in flight per SM.
//
// Same arithmetic contract as qmlp.cuh (AZG_FLAG_EVAL_Q8: exact int8-sliced fixed-point products, oracle/azg_oracle.h),
// different schedule.  ncu on the one-tile-at-a-time kernel (profiles/r1c) showed the SM issuing on 35 % of its cycles: all 16
// warps walk the same phase, so a third of the samples sit at the CTA barriers, in the wait for the MMAs and behind the four
// warps that post-process a finished tile.  Here
//   * a dedicated MMA warp issues every tcgen05.mma; the 16 epilogue warps never issue, they only wait on mbarriers;
//   * two tiles (A, B) of up to 128 rows are in flight and every epilogue warp alternates between them phase by phase, so
//     the MMAs of one tile run under the epilogue arithmetic of the other;
//   * each H x H layer is issued as two N = 64 halves into a 192-column accumulator window per tile (PA | PB | PC, 64
//     columns each): the epilogue of half 0 overlaps the MMAs of half 1, and two tiles fit the 512 TMEM columns
//     (2 x 192 + 2 x 64 columns of scratch for the head partial sums);
//   * a third warpgroup post-processes finished tiles (sum of the head partial sums, softmax / exp of the policy head, scatter
//     into the tree tables): on the epilogue warps that work made one warp of a row group late at every tile and the other
//     three waited for it (12 % of the samples, profiles/r1e);
//   * the only thread barrier left is a 128-thread named barrier among the four warps that share a row group (row maximum);
//   * the tile is a RUN-TIME index everywhere (one copy of the epilogue code: the first version, specialised per tile and
//     layer, was 210 KB of SASS and starved on instruction fetch): the 16 activations a thread produces in half 0 wait for
//     half 1 in the tile's TMEM scratch columns, not in registers.
// Thread (row r = 32*(warp%4) + lane, cq = warp/4) owns outputs j = 32*cq .. 32*cq+31 of row r in every layer (TMEM lane r is
// readable by warps with warp%4 == r/32 only).  Half h of a layer produces the outputs j = 32*cq + 16*h + i, i < 16, of every
// thread: the weight digit planes are stored with their rows permuted (engine.cu pack_weights_q8, qmlp_perm_row) so that
// those are D columns 16*cq + i of the half, and the 16 activations a thread hands to the next layer are one 16-byte k-chunk
// (k/16 = 2*cq + h) of the K-major A operand.
#pragma once
#include "qmlp.cuh"
#include "tree_continuous.cuh"
#include "tree_discrete.cuh"

#define Q2_EPI_THREADS 512
#define Q2_THREADS 768                // 16 epilogue warps + the MMA warpgroup + the post-processing warpgroup (registers rebalanced with setmaxnreg)
#define Q2_MAX_TILES 16               // whole-search kernel: tiles per CTA and launch (engine.cu cuts larger batches into chunks)
#define Q2_PHASE_THREADS 640           // whole-search kernel: the threads that meet between phases (16 epilogue warps + the post-processing warpgroup)
#define Q2_IDESC ((2u << 4) | (1u << 7) | (1u << 10) | ((64u >> 3) << 17) | ((128u >> 4) << 24))  // s8 x s8 -> s32, K-major, N = 64, M = 128
#define Q2_ACC_COLS 192               // accumulator window of a tile: PA | PB | PC, 64 columns each
#define Q2_SCRATCH_COL 384            // head partial sums of tile T: columns 384 + 64 T + 16 cq + c
#define Q2_MAX_PO 16

#define Q2_TAB_BYTES ((FUSED_TAB + 1) * (8 + 8 + 4))  // whole-search kernel: rcp, sqrt and progressive-widening tables in shared memory
__host__ __device__ inline size_t qmlp2_smem_bytes(int NL, int qfl_count, bool fused = false) {
    return (size_t)NL * 3 * QMLP_PLANE + 2 * 3 * QMLP_PLANE + (size_t)qfl_count * 4 + 2 * 4 * 128 * 4 + 1024 + (fused ? Q2_TAB_BYTES : 0);
}
// TSM (trees in shared memory, tree_discrete.cuh ds_step): one tile per CTA, so ONE A-operand slot; behind the tables the rows,
// per-tree scalars, network inputs and leaf words of the CTA's trees
#define Q2_TSM_PER_TREE(R, PO_PAD) ((size_t)(R) * (sizeof(DRow) + 2) + sizeof(STree) + sizeof(float4) + sizeof(int32_t) + 4 * (PO_PAD) * sizeof(float))
__host__ __device__ inline size_t qmlp2_tsm_smem_bytes(int NL, int qfl_count, int trees, int R, int po_pad) {
    return qmlp2_smem_bytes(NL, qfl_count, true) - 3 * QMLP_PLANE + 64 + 16 + (size_t)trees * Q2_TSM_PER_TREE(R, po_pad);
}
// row of the digit planes that holds output j: half h = (j/16)%2, D column of the half = 16*(j/32) + j%16
__host__ __device__ inline int qmlp_perm_row(int j) { return 64 * ((j >> 4) & 1) + 16 * (j >> 5) + (j & 15); }

// The shared-memory descriptors of this kernel differ only in their start-address field: the issuing thread keeps 32-bit low
// words (start address >> 4 | LBO 2048 B) and the MMA assembles the 64-bit operands, so it needs a handful of registers.
#define Q2_DESC_HI ((128u >> 4) | (1u << 14))  // SBO 128 B, descriptor version 1
__device__ __forceinline__ uint32_t q2_desc_lo(uint32_t saddr) { return ((saddr >> 4) & 0x3FFFu) | ((2048u >> 4) << 16); }
__device__ __forceinline__ void umma_i8_n64(uint32_t tmem_d, uint32_t da_lo, uint32_t db_lo, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tmov.b64 da, {%1, %5};\n\tmov.b64 db, {%2, %5};\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], da, db, %3, p;\n\t}" ::"r"(tmem_d),
        "r"(da_lo), "r"(db_lo), "r"(Q2_IDESC), "r"(accumulate), "r"(Q2_DESC_HI)
        : "memory");
}
// one lane of a converged warp (elect.sync): the MMA warp runs its loop with all 32 lanes so that descriptors, window addresses and
// barrier parities are warp-uniform values (uniform registers), and only the tcgen05 instructions themselves sit in the elected branch.
// With the whole loop under `lane == 0` every UTCIMMA was preceded by ~12 instructions moving its operands from the thread's registers
// into uniform ones (R2UR + ELECT ...): ~150 instructions per batch of 12 MMAs issued by one thread at lone-warp latency
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, int32_t* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_ld16f(uint32_t taddr, float* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]), "=f"(v[8]), "=f"(v[9]),
                   "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_st16f(uint32_t taddr, const float* v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
                 "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]), "f"(v[8]), "f"(v[9]), "f"(v[10]),
                 "f"(v[11]), "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15])
                 : "memory");
}
__device__ __forceinline__ void tmem_ld4f(uint32_t taddr, float* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_st4f(uint32_t taddr, float a, float b, float c, float d) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// Phase boundary of the whole-search kernel: every participant arrives (release) and waits for the phase to complete (acquire), so
// the global-memory writes of one phase (tree tables, X) are visible to the readers of the next.  An mbarrier like every other
// cross-role synchronisation of this kernel (a 640-thread named barrier next to the MMA warpgroup parked at barrier 0 computes the
// same results but is reported by compute-sanitizer's synccheck).
__device__ __forceinline__ void phase_sync(uint64_t* bar, uint32_t& parity) {
    mbar_arrive(bar);
    mbar_wait(bar, parity);
    parity ^= 1u;
}
// the same for a warp that has nothing to do for a whole phase (the post-processing warps during the tree phase): it sleeps between
// polls instead of competing with the tree warps of its scheduler for issue slots
__device__ __forceinline__ void phase_sync_idle(uint64_t* bar, uint32_t& parity) {
    mbar_arrive(bar);
#ifndef AZG_NO_IDLE_SLEEP
    while (!mbar_try_wait(bar, parity)) __nanosleep(256);
#else
    mbar_wait(bar, parity);
#endif
    parity ^= 1u;
}

// per-CTA constants of the epilogue warps
struct Q2Ctx {
    const float* W0;     // [S][H] layer-0 weights, k-major
    const float* b0;     // [H]
    const float2* cwb;   // [NL][H] (cw[j], bias[j])
    const float* Wh;     // [H][PO_PAD]
    const float* bh;     // [PO_PAD]
    float* pmax;         // [2][4][128]
    int8_t* sA;          // [2][3][QMLP_PLANE]
    uint64_t *full, *ready, *freeb, *hfull;
    uint32_t tb;         // TMEM base
    int r, lg, cq;
};

// row maximum over the four column quarters -> scale -> digits of this thread's two k-chunks -> shared memory -> "ready"
__device__ __forceinline__ float q2_quantise_store(const Q2Ctx& c, int T, bool wact, const float* a0, const float* a1, float pm) {
    float cx = 0.0f;
    if (wact) {
        float* pmx = c.pmax + T * 512;
        pmx[c.cq * 128 + c.r] = pm;
        group_sync(1 + c.lg, 128);
        const float m = fmaxf(fmaxf(pmx[c.r], pmx[128 + c.r]), fmaxf(pmx[256 + c.r], pmx[384 + c.r]));
        const int e = q8_exponent(m);
        const float sx = __uint_as_float((uint32_t)(276 - e) << 23);  // 2^(149-e)
        cx = __uint_as_float((uint32_t)(e - 22) << 23);               // 2^(e-149)
        int8_t* sAT = c.sA + T * 3 * QMLP_PLANE;
        q8_store16(a0, sx, sAT, c.cq * 2, c.r);
        q8_store16(a1, sx, sAT, c.cq * 2 + 1, c.r);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes of A -> visible to the tensor core
    }
    mbar_arrive(c.ready + T);
    return cx;
}

// layer 0 (S -> H) in FP32 FMA on this thread's 32 outputs, then quantise
template <int S, int ACT>
__device__ __forceinline__ float q2_layer0(const Q2Ctx& c, const MlpParams& p, int T, bool wact, int gr, bool valid) {
    float a[32];
    float pm = 0.0f;
    if (wact) {
        float x[S];
#pragma unroll
        for (int s = 0; s < S; ++s) x[s] = 0.0f;
        if (valid) {
            if constexpr (S > 4) {  // Acrobot: 6 inputs in two float4 per leaf (the tree writes xstride 8)
                if (p.xstride == 8) {
                    const float4 v = *reinterpret_cast<const float4*>(p.X + (size_t)gr * 8), w = *reinterpret_cast<const float4*>(p.X + (size_t)gr * 8 + 4);
                    x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w; x[4] = w.x; x[5] = w.y;
                } else {
#pragma unroll
                    for (int s = 0; s < S; ++s) x[s] = p.X[(size_t)gr * p.xstride + s];
                }
            } else if (p.xstride == 4) {
                const float4 v = *reinterpret_cast<const float4*>(p.X + (size_t)gr * 4);
                x[0] = v.x; x[1] = v.y;
                if constexpr (S > 2) x[2] = v.z;
                if (S > 3) x[S - 1] = v.w;
            } else {
#pragma unroll
                for (int s = 0; s < S; ++s) x[s] = p.X[(size_t)gr * p.xstride + s];
            }
        }
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
            const int j = c.cq * 32 + i;
            float2 acc = *reinterpret_cast<const float2*>(c.b0 + j);
#pragma unroll
            for (int s = 0; s < S; ++s) acc = __ffma2_rn(make_float2(x[s], x[s]), *reinterpret_cast<const float2*>(c.W0 + s * 128 + j), acc);
            const float2 e = mlp_act2<ACT>(acc);
            a[i] = e.x; a[i + 1] = e.y;
            pm = fmaxf(pm, fmaxf(fabsf(e.x), fabsf(e.y)));
        }
    }
    return q2_quantise_store(c, T, wact, a, a + 16, pm);
}

// heads: partial FMA chains over this thread's 32 activations -> the tile's TMEM scratch -> "hfull" (the post-processing warps
// sum the four partials of every output and finish the row)
__device__ __forceinline__ void q2_heads(const Q2Ctx& c, const MlpParams& p, int T, bool wact, const float* a0, const float* a1) {
    if (wact) {
        const uint32_t lane_base = c.tb + ((uint32_t)(c.lg * 32) << 16) + Q2_SCRATCH_COL + T * 64;
#pragma unroll 1
        for (int c4 = 0; c4 < p.PO_PAD / 4; ++c4) {
            float2 lo = make_float2(0.0f, 0.0f), hi = make_float2(0.0f, 0.0f);
            const float* wp = c.Wh + (c.cq * 32) * p.PO_PAD + c4 * 4;
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const float4 w4 = *reinterpret_cast<const float4*>(wp + i * p.PO_PAD);
                const float ai = i < 16 ? a0[i & 15] : a1[i & 15];
                const float2 av = make_float2(ai, ai);
                lo = __ffma2_rn(av, make_float2(w4.x, w4.y), lo);
                hi = __ffma2_rn(av, make_float2(w4.z, w4.w), hi);
            }
            tmem_st4f(lane_base + c.cq * 16 + c4 * 4, lo.x, lo.y, hi.x, hi.y);
        }
        tmem_wait_st();
    }
    tc_fence_before();
    mbar_arrive(c.hfull + T);
}

// TSM: the same chains, partial sums into shared memory ([4 quarters][PO_PAD][trees]); the tree phase sums them and finishes the row
__device__ __forceinline__ void q2_heads_tsm(const Q2Ctx& c, const MlpParams& p, bool active, const float* a0, const float* a1, float* part, int ntrees) {
    if (active) {
#pragma unroll 1
        for (int c4 = 0; c4 < p.PO_PAD / 4; ++c4) {
            float2 lo = make_float2(0.0f, 0.0f), hi = make_float2(0.0f, 0.0f);
            const float* wp = c.Wh + (c.cq * 32) * p.PO_PAD + c4 * 4;
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const float4 w4 = *reinterpret_cast<const float4*>(wp + i * p.PO_PAD);
                const float ai = i < 16 ? a0[i & 15] : a1[i & 15];
                const float2 av = make_float2(ai, ai);
                lo = __ffma2_rn(av, make_float2(w4.x, w4.y), lo);
                hi = __ffma2_rn(av, make_float2(w4.z, w4.w), hi);
            }
            float* d = part + (size_t)(c.cq * p.PO_PAD + c4 * 4) * ntrees + c.r;
            d[0] = lo.x; d[ntrees] = lo.y; d[2 * ntrees] = hi.x; d[3 * ntrees] = hi.y;
        }
    }
}

// post-processing warp of row group lg: one thread per row of the tile in slot T (ROW3: mlp_finish_row)
template <bool ROW3>
__device__ __forceinline__ void q2_finish_tile(const MlpParams& p, uint32_t tb, const float* bh, int lg, int T, bool need, int gr, int leafw,
                                               double lr, uint64_t* hfree, uint32_t& nev, int& ev_row) {
    const uint32_t lane_base = tb + ((uint32_t)(lg * 32) << 16) + Q2_SCRATCH_COL + T * 64;
    float out[Q2_MAX_PO];
#pragma unroll  // static indices: out[] stays in registers
    for (int c4 = 0; c4 < Q2_MAX_PO / 4; ++c4) {
        if (c4 < p.PO_PAD / 4) {
            float q0[4], q1[4], q2[4], q3[4];
            tmem_ld4f(lane_base + c4 * 4, q0);
            tmem_ld4f(lane_base + 16 + c4 * 4, q1);
            tmem_ld4f(lane_base + 32 + c4 * 4, q2);
            tmem_ld4f(lane_base + 48 + c4 * 4, q3);
            tmem_wait_ld();
#pragma unroll
            for (int i = 0; i < 4; ++i)
                out[c4 * 4 + i] = __fadd_rn(__fadd_rn(__fadd_rn(q0[i], q1[i]), __fadd_rn(q2[i], q3[i])), bh[c4 * 4 + i]);
        } else {
#pragma unroll
            for (int i = 0; i < 4; ++i) out[c4 * 4 + i] = 0.0f;
        }
    }
    tc_fence_before();
    mbar_arrive(hfree + T);  // the scratch columns may be reused (half-0 activations of the next tile in this slot)
    if (need) {
        mlp_finish_row<ROW3>(p, gr, leafw, lr, out[0], out + 1);
        ++nev;
        ev_row = gr;
    }
}

// ---- evaluation of ONE thin tile (at most 32 rows) by all 16 epilogue warps: "replicated rows" (whole-search kernel, TSM) -------------
// A tile of 28 rows fills one TMEM lane group, and a lane group is readable by the warps with warp % 4 == group only -- the four warps
// of ONE scheduler (evaluation timeline, profiles/README.md r2s: 3040 cycles for layer 0 + quantisation, 1900 for the accumulator
// conversion, 1800 for quantise / heads per simulation on that scheduler, three schedulers idle).  Here row r of the tile is written
// into the A operand FOUR times, at rows r, 32 + r, 64 + r, 96 + r, so every lane group holds every tree after the M = 128 MMAs (which
// cost the same whatever the rows hold), and the 16 threads (lane group lg, column quarter cq) of a tree split its columns: thread
// (lg, cq) owns the outputs j = 32 cq + 16 h + 4 lg + i (half h < 2, i < 4), a quarter of what thread (cq) owns in the ordinary
// schedule.  Per-element arithmetic is unchanged; the row maximum is exchanged through shared memory by all 16 warps; the heads keep
// the contract's summation order (four chains over 32 consecutive activations): the last layer's activations go through shared memory
// (they alias the A operand, dead by then) and the chain of quarter q runs on warp q -- a different scheduler each --, its partial
// sums go where the tree phase expects them (SmTrees::part).
__device__ __forceinline__ void tmem_ld4i(uint32_t taddr, int32_t* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(taddr) : "memory");
}
#define Q2_REP_BAR 5  // named barrier of the 16 epilogue warps (ids 1..4 are the row groups')
// row maximum over the tree's 16 threads -> scale -> digits of this thread's 8 activations into the four row replicas -> "ready"
__device__ __forceinline__ float q2_rep_quantise_store(const Q2Ctx& c, const float* a, float pm, int r) {
    float* pmx = c.pmax;  // [16][32]
    pmx[(c.lg * 4 + c.cq) * 32 + r] = pm;
    group_sync(Q2_REP_BAR, Q2_EPI_THREADS);
    float m = 0.0f;
#pragma unroll
    for (int w = 0; w < 16; ++w) m = fmaxf(m, pmx[w * 32 + r]);
    const int e = q8_exponent(m);
    const float sx = __uint_as_float((uint32_t)(276 - e) << 23);  // 2^(149-e)
    const float cx = __uint_as_float((uint32_t)(e - 22) << 23);   // 2^(e-149)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        uint32_t t[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) t[i] = (q8_quant(__fmul_rn(a[4 * h + i], sx)) + 0x8080u) ^ 0x8080u;
        const uint32_t lo01 = __byte_perm(t[0], t[1], 0x5140), lo23 = __byte_perm(t[2], t[3], 0x5140);
        const uint32_t hi01 = __byte_perm(t[0], t[1], 0x0062), hi23 = __byte_perm(t[2], t[3], 0x0062);
        const uint32_t wlo = __byte_perm(lo01, lo23, 0x5410), wmid = __byte_perm(lo01, lo23, 0x7632), whi = __byte_perm(hi01, hi23, 0x5410);
        int8_t* d = c.sA + (2 * c.cq + h) * 2048 + r * 16 + 4 * c.lg;  // k-chunk (32 cq + 16 h) / 16, bytes 4 lg .. 4 lg + 3 of the row's 16
#pragma unroll
        for (int m4 = 0; m4 < 4; ++m4) {
            *reinterpret_cast<uint32_t*>(d + m4 * 512) = whi;
            *reinterpret_cast<uint32_t*>(d + m4 * 512 + QMLP_PLANE) = wmid;
            *reinterpret_cast<uint32_t*>(d + m4 * 512 + 2 * QMLP_PLANE) = wlo;
        }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes of A -> visible to the tensor core
    mbar_arrive(c.ready);
    return cx;
}
// one evaluation of the tile in slot 0 (rows row0 .. row0 + nv - 1, nv <= 32); sact: [128][32] activations of the last layer (aliases the
// A operand); part: [4][PO_PAD][nv] head partial sums for the tree phase
template <int S, int ACT, int NL>
__device__ __forceinline__ void q2_eval_rep(const Q2Ctx& c, const MlpParams& p, int nv, int row0, int lane, uint32_t& fullph, float* sact, float* part) {
    const int r = lane;
    const int jb = 32 * c.cq + 4 * c.lg;  // outputs jb + 16 h + i
    float a[8];
    float pm = 0.0f;
    {
        float x[S];
#pragma unroll
        for (int s = 0; s < S; ++s) x[s] = 0.0f;
        if (r < nv) {
            if constexpr (S > 4) {  // Acrobot: xstride 8 in the whole-search kernel
                const float4 v = *reinterpret_cast<const float4*>(p.X + (size_t)(row0 + r) * 8), w = *reinterpret_cast<const float4*>(p.X + (size_t)(row0 + r) * 8 + 4);
                x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w; x[4] = w.x; x[5] = w.y;
            } else {
                const float4 v = *reinterpret_cast<const float4*>(p.X + (size_t)(row0 + r) * 4);  // xstride 4 in the whole-search kernel
                x[0] = v.x; x[1] = v.y;
                if constexpr (S > 2) x[2] = v.z;
                if (S > 3) x[S - 1] = v.w;
            }
        }
#pragma unroll
        for (int k = 0; k < 8; k += 2) {
            const int j = jb + 16 * (k >> 2) + (k & 3);
            float2 acc = *reinterpret_cast<const float2*>(c.b0 + j);
#pragma unroll
            for (int s = 0; s < S; ++s) acc = __ffma2_rn(make_float2(x[s], x[s]), *reinterpret_cast<const float2*>(c.W0 + s * 128 + j), acc);
            const float2 e = mlp_act2<ACT>(acc);
            a[k] = e.x; a[k + 1] = e.y;
            pm = fmaxf(pm, fmaxf(fabsf(e.x), fabsf(e.y)));
        }
    }
    float cx = q2_rep_quantise_store(c, a, pm, r);
    const uint32_t ta = c.tb + ((uint32_t)(c.lg * 32) << 16) + 16 * c.cq + 4 * c.lg;
#pragma unroll 1
    for (int l = 0; l < NL; ++l) {
        pm = 0.0f;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            mbar_wait(c.full, fullph & 1u);
            fullph ^= 1u;
            tc_fence_after();
            int32_t pa[4], pb[4], pc[4];
            tmem_ld4i(ta, pa);
            tmem_ld4i(ta + 64, pb);
            tmem_ld4i(ta + 128, pc);
            tmem_wait_ld();
            tc_fence_before();
            if (h == 0) mbar_arrive(c.freeb);  // the window may be overwritten by the MMAs of half 1
            const float2* cb = c.cwb + l * 128 + jb + 16 * h;
#pragma unroll
            for (int i = 0; i < 4; i += 2) {
                const float4 sb = *reinterpret_cast<const float4*>(cb + i);  // (cw, bias) of outputs i, i+1
                float u0 = __int2float_rn(pa[i] * 256 + pb[i]);                 // = fma(PA, 256, PB), see the ordinary schedule below
                float u1 = __int2float_rn(pa[i + 1] * 256 + pb[i + 1]);
                u0 = __fmaf_rn(u0, 256.0f, q8_i2f_23(pc[i]));
                u1 = __fmaf_rn(u1, 256.0f, q8_i2f_23(pc[i + 1]));
                const float2 y = make_float2(__fmaf_rn(u0, __fmul_rn(cx, sb.x), sb.y), __fmaf_rn(u1, __fmul_rn(cx, sb.z), sb.w));
                const float2 ev = mlp_act2<ACT>(y);
                a[4 * h + i] = ev.x; a[4 * h + i + 1] = ev.y;
                pm = fmaxf(pm, fmaxf(fabsf(ev.x), fabsf(ev.y)));
            }
        }
        if (l + 1 < NL) cx = q2_rep_quantise_store(c, a, pm, r);
    }
    // heads: the activations of the last layer through shared memory, the chain of quarter q on warp q
#pragma unroll
    for (int k = 0; k < 8; ++k) sact[(jb + 16 * (k >> 2) + (k & 3)) * 32 + r] = a[k];
    group_sync(Q2_REP_BAR, Q2_EPI_THREADS);
    if (c.cq == 0 && r < nv) {
        const int q = c.lg;
#pragma unroll 1
        for (int c4 = 0; c4 < p.PO_PAD / 4; ++c4) {
            float2 lo = make_float2(0.0f, 0.0f), hi = make_float2(0.0f, 0.0f);
            const float* wp = c.Wh + (q * 32) * p.PO_PAD + c4 * 4;
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const float4 w4 = *reinterpret_cast<const float4*>(wp + i * p.PO_PAD);
                const float ai = sact[(q * 32 + i) * 32 + r];
                const float2 av = make_float2(ai, ai);
                lo = __ffma2_rn(av, make_float2(w4.x, w4.y), lo);
                hi = __ffma2_rn(av, make_float2(w4.z, w4.w), hi);
            }
            float* d = part + (size_t)(q * p.PO_PAD + c4 * 4) * nv + r;
            d[0] = lo.x; d[nv] = lo.y; d[2 * nv] = hi.x; d[3 * nv] = hi.y;
        }
    }
}

// FUSED = false: one leaf evaluation of p.n rows (one launch per simulation, engine.cu enqueue_search).
// FUSED = true: the WHOLE SEARCH of the continuous tree for the trees [chunk_begin, chunk_end) in one persistent launch.
//   Trees never interact, so nothing needs a grid-wide barrier between simulations: a CTA owns its trees for the whole search
//   and alternates two phases, n_sims + 1 times: (1) the evaluation of all its tiles, exactly as above; (2) a TREE PHASE in which
//   the 16 epilogue warps run one thread per tree: backup of the finished simulation, descent + expansion of the next (c_step,
//   tree_continuous.cuh -- the body of k_step_continuous), next network input into X.  Two phase boundaries (an mbarrier all 640 of them arrive at and wait on) separate the
//   phases (epilogue warps + post-processing warpgroup; the MMA warp only follows its mbarriers).  What this buys over one launch
//   per kernel and simulation: weights, TMEM and barriers are set up once per search instead of once per simulation (~10 us of
//   ramp per evaluation launch, tools/step_scaling.py), no launch gaps, and the 148 CTAs drift out of phase, so the tree phases
//   of some SMs overlap the evaluations of others and the HBM traffic of the tree walk is spread over the whole simulation
//   instead of arriving in one burst.  The first version (git history, profiles/README.md r1f) overlapped the two phases INSIDE
//   an SM with two dedicated tree warpgroups; at 48 registers per tree thread and with both code paths fighting for the
//   instruction cache it reached 80 us per simulation against 74 us for separate launches.
// TSM (FUSED, discrete tree, thin batches): the CTA's trees live in shared memory for the whole search (tree_discrete.cuh ds_step).
// ENV (env.cuh): CartPole = the discrete tree, Pendulum | MountainCarContinuous = the continuous tree stepping that env; its S is the
// width of layer 0.
template <class ENV, int ACT, int NL, bool FUSED, bool TSM = false>
__global__ void __launch_bounds__(Q2_THREADS, 1)
k_qmlp2(const MlpParams p_in, const TreeParams tp, const int n_sims, const int chunk_begin, const int chunk_end) {
    constexpr int S = ENV::S;
    static_assert(!TSM || (FUSED && env::actions_of<ENV>() == 2), "trees in shared memory: whole-search kernel of the two-action discrete tree");
    extern __shared__ __align__(1024) uint8_t qsm_raw[];
    __shared__ __align__(8) uint64_t wbar, full[2], ready[2], freeb[2], hfull[2], hfree[2], phase_bar;
    __shared__ uint32_t tmem_base_s;
    __shared__ DsCtx s_dsctx;  // TSM: context of the tree phase (tree_discrete.cuh ds_phase)
    __shared__ unsigned long long s_dsprof[8];
    // round up to 1024 B with an OFFSET on the shared pointer: a round trip through uintptr_t loses the address space and every
    // access below becomes a generic LD/ST (long-scoreboard latency) instead of LDS/STS
    uint8_t* qsm = qsm_raw + ((1024u - (smem_u32(qsm_raw) & 1023u)) & 1023u);
    int8_t* sB = reinterpret_cast<int8_t*>(qsm);                     // [NL][3][8][128][16], rows permuted
    int8_t* sA = sB + (size_t)NL * 3 * QMLP_PLANE;                   // [2][3][8][128][16]
    float* fl = reinterpret_cast<float*>(sA + (TSM ? 1 : 2) * 3 * QMLP_PLANE);   // W0t[S][H], b0[H], NL x (cw, bias)[H], Wh[H][PO_PAD], bh[PO_PAD]
    float* pmax = fl + p_in.qfl_count;                               // [2][4][128]
    double* s_rcp = reinterpret_cast<double*>(pmax + 2 * 4 * 128);   // whole-search kernel: [FUSED_TAB + 1] each
    double* s_sq = s_rcp + FUSED_TAB + 1;
    int32_t* s_pw = reinterpret_cast<int32_t*>(s_sq + FUSED_TAB + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    // this CTA's contiguous row range, cut into an even number of equal tiles of at most 128 rows
    const int first = FUSED ? chunk_begin : 0, last = FUSED ? chunk_end : p_in.n;
    const int per = (last - first + gridDim.x - 1) / gridDim.x;
    const int row_begin = first + blockIdx.x * per;
    const int row_end = min(row_begin + per, last);
    const int n_evals = FUSED ? n_sims + 1 : 1;  // evaluations per tile: the root + one per simulation
    if (row_begin >= row_end) return;
    const int nrows = row_end - row_begin;
    int ntiles = (nrows + 127) / 128;
    if (ntiles > 1) ntiles = (ntiles + 1) & ~1;
    // TSM: shared-memory tables of the CTA's trees behind the lookup tables.  The evaluation reads its network inputs from them through a
    // patched copy of the parameter block (a generic address that points into shared memory) and leaves the head's partial sums in
    // `part`; the tree phase finishes the rows itself (tree_discrete.cuh ds_step), so the post-processing warps only keep the phase
    // barriers' count
    SmTrees smt;
    {
        uint8_t* tbase = reinterpret_cast<uint8_t*>(s_pw + FUSED_TAB + 1);
        tbase += (64u - (smem_u32(tbase) & 63u)) & 63u;
        smt.rows = reinterpret_cast<DRow*>(tbase);
        smt.st = reinterpret_cast<STree*>(smt.rows + (size_t)(TSM ? nrows : 0) * tp.R);
        smt.X = reinterpret_cast<float4*>(smt.st + (TSM ? nrows : 0));
        smt.leaf = reinterpret_cast<int32_t*>(smt.X + (TSM ? nrows : 0));
        smt.path = reinterpret_cast<uint16_t*>(smt.leaf + (TSM ? nrows : 0));
        uint8_t* pbase = reinterpret_cast<uint8_t*>(smt.path + (size_t)(TSM ? nrows : 0) * tp.R);
        pbase += (16u - (smem_u32(pbase) & 15u)) & 15u;
        smt.part = reinterpret_cast<float*>(pbase);
    }
    MlpParams p_tsm;
    if (TSM) {
        p_tsm = p_in;
        p_tsm.X = reinterpret_cast<const float*>(smt.X) - (ptrdiff_t)row_begin * 4;
    }
    const MlpParams& p = TSM ? p_tsm : p_in;
    if (TSM && tid == 0) {
        DsCtx cx;
        cx.sm = smt;
        cx.dstate = tp.dstate + (size_t)row_begin * tp.R * 4;
        cx.err = tp.err;
        cx.rcp = s_rcp; cx.sq = s_sq;
        cx.gamma = tp.gamma; cx.epsilon = tp.epsilon; cx.c_uct = tp.c_uct;
        cx.reward_step = tp.reward_step; cx.reward_terminal = tp.reward_terminal;
        const uint64_t seed = __ldg(tp.seedp);
        cx.k0 = (uint32_t)seed; cx.k1 = (uint32_t)(seed >> 32);
        cx.tree0 = tree_base(tp) + row_begin;
        cx.tabn = FUSED_TAB; cx.R = tp.R; cx.puct_f32 = tp.puct_f32; cx.ntrees = nrows;
        // a group of lpt consecutive lanes per tree.  Measured at 28 trees per CTA (profiles/README.md r2n): lpt = 16 (14 warps) 320,
        // lpt = 8 (7 warps) 337, lpt = 4 (4 warps) 318 M sims/s -- fewer warps issue fewer instructions in total (both halves of
        // a warp share one stream), more lanes per tree shorten the backup and the draw generation
        cx.lpt = nrows <= 64 ? 8 : 4;
        cx.po_pad = p_in.PO_PAD;
        cx.bh = fl + S * 128 + 128 + NL * 2 * 128 + 128 * p_in.PO_PAD;
#ifdef AZG_TSM_LPT
        cx.lpt = AZG_TSM_LPT;
#endif
        cx.prof = s_dsprof;
        for (int k = 0; k < 8; ++k) s_dsprof[k] = 0;
        s_dsctx = cx;
    }
    // full tiles first, the remainder in the last one(s): epilogue work is spent per 32-row group, so 443 rows cost 14 row groups
    // as 128 + 128 + 128 + 59 against 16 as four tiles of 111 (the warps of the empty row groups leave their issue slots to the others)
    const int th = 128;

    if (tid == 0) {
        mbar_init(&wbar, 1);
        mbar_init(&phase_bar, Q2_PHASE_THREADS);
        for (int T = 0; T < 2; ++T) {
            mbar_init(&full[T], 1);
            mbar_init(&ready[T], Q2_EPI_THREADS);
            mbar_init(&freeb[T], Q2_EPI_THREADS);
            mbar_init(&hfull[T], Q2_EPI_THREADS);
            mbar_init(&hfree[T], 128);
        }
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "n"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tb = tmem_base_s;
    if (tid == 0) {
        const uint32_t bytesB = (uint32_t)NL * 3 * QMLP_PLANE, bytesF = (uint32_t)p.qfl_count * 4u;
        mbar_expect_tx(&wbar, bytesB + bytesF);
        for (uint32_t o = 0; o < bytesB; o += 32768u) bulk_g2s(sB + o, p.qdigits + o, min(32768u, bytesB - o), &wbar);
        bulk_g2s(fl, p.qfl, bytesF, &wbar);
    }
    if (FUSED) {
        for (int i = tid; i <= FUSED_TAB; i += blockDim.x) {
            s_rcp[i] = tp.rcp_tab[i];
            s_sq[i] = tp.sqrt_tab[i];
            s_pw[i] = (tp.pw_table && i < p.R) ? tp.pw_table[i] : 0;  // continuous only; the table has max_rollouts + 2 = R entries
        }
        __syncthreads();
    }
    mbar_wait(&wbar, 0);

    if (warp >= 20) {
        // ---- post-processing warpgroup: warp 20 + lg finishes the rows of row group lg, tile after tile
        asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
        const int lg = warp & 3, r = lg * 32 + lane;
        const float* bh = fl + S * 128 + 128 + NL * 2 * 128 + 128 * p.PO_PAD;
        uint32_t hph = 0, nev = 0;
        int ev_row = 0;
        uint32_t pph = 0;  // parity of the next phase boundary
        if (FUSED) phase_sync(&phase_bar, pph);  // the roots are initialised (c_init)
#pragma unroll 1
        for (int s = 0; s < n_evals; ++s) {
#pragma unroll 1
        for (int t = 0; t < (TSM ? 0 : ntiles); ++t) {  // TSM: the tree phase finishes the rows itself (tree_discrete.cuh ds_step)
            const int T = t & 1;
            const int row0 = row_begin + t * th;
            const int nv = max(0, min(th, row_end - row0));
            const int gr = row0 + r;
            bool need = r < nv;
            int leafw = 0;
            double lr = 0.0;
            if (need && p.mode == 0) {  // loaded before the wait: the latency hides under the tile's evaluation
                if (p.variant == 1) {
                    const uint4 c0 = p.ctl[gr], c1 = p.ctl[(size_t)p.BS + gr];
                    leafw = (int)c0.z;
                    lr = __hiloint2double((int)c1.w, (int)c1.z);
                } else {
                    leafw = p.leaf[gr];
                }
                need = (leafw & LEAF_EVAL) != 0;
            }
            mbar_wait(&hfull[T], (hph >> T) & 1u);
            hph ^= 1u << T;
            tc_fence_after();
            if (lg * 32 < nv) q2_finish_tile<env::row3<ENV>()>(p, tb, bh, lg, T, need, gr, leafw, lr, hfree, nev, ev_row);
            else mbar_arrive(&hfree[T]);
        }
        if (FUSED) {
            phase_sync(&phase_bar, pph);  // every row of this evaluation is finished: the tree phase may start
            phase_sync_idle(&phase_bar, pph);  // the tree phase is over: leaf words and X of the next simulation are in place
        }
        }
        if (nev && p.mode == 0) p.evals[ev_row] += nev;  // only the total over trees is reported (azg_get_counters)
    } else if (warp >= 16) {
        // ---- MMA warpgroup: gives its registers to the epilogue warps; one thread issues, in the order the epilogue warps consume
        asm volatile("setmaxnreg.dec.sync.aligned.u32 24;");
        if (warp == 16) {
            uint32_t rph = 0, fph = 0;  // bit T: parity of the next wait on ready[T] / freeb[T]
#pragma unroll 1
            for (int s = 0; s < n_evals; ++s)
            for (int t0 = 0; t0 < ntiles; t0 += 2) {
                const int nt = min(2, ntiles - t0);
#pragma unroll 1
                for (int l = 0; l < NL; ++l) {
#pragma unroll 1
                    for (int hT = 0; hT < 2 * nt; ++hT) {
                        const int h = hT >> (nt - 1), T = hT & (nt - 1);  // nt is 1 or 2
                        if (h == 0) { mbar_wait(&ready[T], (rph >> T) & 1u); rph ^= 1u << T; }
                        else { mbar_wait(&freeb[T], (fph >> T) & 1u); fph ^= 1u << T; }
                        tc_fence_after();
                        // low descriptor words: +1024 per digit plane (16 KB), +256 per k-step of 32 (4 KB)
                        const uint32_t aH = q2_desc_lo(smem_u32(sA) + (uint32_t)T * 3 * QMLP_PLANE), aM = aH + 1024, aL = aH + 2048;
                        const uint32_t bH = q2_desc_lo(smem_u32(sB) + (uint32_t)l * 3 * QMLP_PLANE + (uint32_t)h * 1024u), bM = bH + 1024, bL = bH + 2048;
                        const uint32_t acc = tb + T * Q2_ACC_COLS;
                        if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < 4; ++k) umma_i8_n64(acc, aH + k * 256, bH + k * 256, k > 0);        // PA = xh*wh
#pragma unroll
                        for (int k = 0; k < 4; ++k) umma_i8_n64(acc + 64, aH + k * 256, bM + k * 256, k > 0);   // PB = xh*wm
#pragma unroll
                        for (int k = 0; k < 4; ++k) umma_i8_n64(acc + 64, aM + k * 256, bH + k * 256, 1);       //    + xm*wh
#pragma unroll
                        for (int k = 0; k < 4; ++k) umma_i8_n64(acc + 128, aH + k * 256, bL + k * 256, k > 0);  // PC = xh*wl
#pragma unroll
                        for (int k = 0; k < 4; ++k) umma_i8_n64(acc + 128, aM + k * 256, bM + k * 256, 1);      //    + xm*wm
#pragma unroll
                        for (int k = 0; k < 4; ++k) umma_i8_n64(acc + 128, aL + k * 256, bH + k * 256, 1);      //    + xl*wh
                        umma_commit(&full[T]);
                        }
                        __syncwarp();
                    }
                }
            }
        }
    } else {
        // ---- epilogue warps
        asm volatile("setmaxnreg.inc.sync.aligned.u32 104;");  // 512 x 104 + 128 x 24 + 128 x 40 = 768 x 80, the CTA's pool at launch
        Q2Ctx c;
        c.W0 = fl;
        c.b0 = fl + S * 128;
        c.cwb = reinterpret_cast<const float2*>(fl + S * 128 + 128);
        c.Wh = fl + S * 128 + 128 + NL * 2 * 128;
        c.bh = c.Wh + 128 * p.PO_PAD;
        c.pmax = pmax;
        c.sA = sA;
        c.full = full; c.ready = ready; c.freeb = freeb; c.hfull = hfull;
        c.tb = tb;
        c.lg = warp & 3; c.cq = warp >> 2;
        c.r = c.lg * 32 + lane;
        long long cyc_tree = 0, cyc_sync = 0;
        const long long cyc_begin = clock64();
        const Tabs tabs = {s_pw, s_rcp, s_sq, FUSED_TAB};
        uint32_t pph = 0;  // parity of the next phase boundary
        if (FUSED) {  // MCTSContinuous.initialize_search for every tree of the CTA
            for (int i = tid; i < nrows; i += Q2_EPI_THREADS) {
                if (TSM) ds_init(tp, smt, i, row_begin + i);
                else if constexpr (ENV::DISCRETE) d_init<ENV>(tp, row_begin + i);
                else c_init<ENV>(tp, row_begin + i);
            }
            phase_sync(&phase_bar, pph);
        }
#ifdef AZG_EVAL_PROF
        // timeline of the evaluation phase on epilogue thread 0: [0] layer 0 + quantise, [1] wait for the MMAs, [2] accumulator loads +
        // conversion + activation, [3] stash / quantise / heads, [4] wait for the post-processing warps, [5] tree phase
        long long ep_last = clock64();
#define EP_STAMP(k) do { const long long _t = clock64(); if (tid == 0) s_dsprof[k] += (unsigned long long)(_t - ep_last); ep_last = _t; } while (0)
        if (!TSM && tid == 0) for (int k = 0; k < 8; ++k) s_dsprof[k] = 0;
#else
#define EP_STAMP(k)
#endif
        uint32_t fullph = 0;  // bit T: parity of the next wait on full[T]
        uint32_t hfph = 0;    // bit T: parity of the next wait on hfree[T]
#pragma unroll 1
        for (int s = 0; s < n_evals; ++s) {
        if (TSM && nrows <= 32) {
            q2_eval_rep<S, ACT, NL>(c, p, nrows, row_begin, lane, fullph, reinterpret_cast<float*>(sA), smt.part);
            EP_STAMP(0);
        } else
#pragma unroll 1
        for (int t0 = 0; t0 < ntiles; t0 += 2) {
            const int nt = min(2, ntiles - t0);
            float cx0 = 0.0f, cx1 = 0.0f;  // per slot (slot T holds tile t0 + T): scale of the current layer's input
#pragma unroll 1
            for (int T = 0; T < nt; ++T) {
                const int row0 = row_begin + (t0 + T) * th;
                const int nv = max(0, min(th, row_end - row0));
                const float cx = q2_layer0<S, ACT>(c, p, T, c.lg * 32 < nv, row0 + c.r, c.r < nv);
                if (T == 0) cx0 = cx; else cx1 = cx;
            }
            EP_STAMP(0);
#pragma unroll 1
            for (int step = 0; step < NL * 2 * nt; ++step) {
                // step -> (layer, half, tile), tile fastest; nt is 1 or 2
                const int sh = nt - 1, T = step & sh, h = (step >> sh) & 1, l = step >> (sh + 1);
                const int row0 = row_begin + (t0 + T) * th;
                const int nv = max(0, min(th, row_end - row0));
                const bool wact = c.lg * 32 < nv;
                const float cx = T ? cx1 : cx0;
                mbar_wait(full + T, (fullph >> T) & 1u);
                fullph ^= 1u << T;
                tc_fence_after();
                EP_STAMP(1);
                const uint32_t lane_base = tb + ((uint32_t)(c.lg * 32) << 16);
                const uint32_t stash = lane_base + Q2_SCRATCH_COL + T * 64 + c.cq * 16;
                float v[16];
                float pm = 0.0f;
                if (wact) {
                    const float2* cb = c.cwb + l * 128 + c.cq * 32 + 16 * h;
                    const uint32_t ta = lane_base + T * Q2_ACC_COLS + c.cq * 16;
                    int32_t pa[16], pb[16], pc[16];
                    tmem_ld16(ta, pa);
                    tmem_ld16(ta + 64, pb);
                    tmem_ld16(ta + 128, pc);
                    tmem_wait_ld();
                    tc_fence_before();
                    if (h == 0) mbar_arrive(freeb + T);  // the window may be overwritten by the MMAs of half 1
#pragma unroll
                    for (int i = 0; i < 16; i += 2) {
                        const float4 sb = *reinterpret_cast<const float4*>(cb + i);  // (cw, bias) of outputs i, i+1
#ifdef AZG_DEQ_FLOAT
                        float u0 = __fmaf_rn(q8_i2f_22(pa[i]), 256.0f, q8_i2f_22(pb[i]));
                        float u1 = __fmaf_rn(q8_i2f_22(pa[i + 1]), 256.0f, q8_i2f_22(pb[i + 1]));
#else
                        // fma(PA, 256, PB) of the contract is the correctly rounded value of the integer PA * 256 + PB (both terms are exact in f32,
                        // |PA * 256 + PB| < 2^31): form it in integer arithmetic and convert once -- 2 instructions instead of 5, none on the FMA pipe
                        float u0 = __int2float_rn(pa[i] * 256 + pb[i]);
                        float u1 = __int2float_rn(pa[i + 1] * 256 + pb[i + 1]);
#endif
                        u0 = __fmaf_rn(u0, 256.0f, q8_i2f_23(pc[i]));
                        u1 = __fmaf_rn(u1, 256.0f, q8_i2f_23(pc[i + 1]));
                        const float2 y = make_float2(__fmaf_rn(u0, __fmul_rn(cx, sb.x), sb.y), __fmaf_rn(u1, __fmul_rn(cx, sb.z), sb.w));
                        const float2 ev = mlp_act2<ACT>(y);
                        v[i] = ev.x; v[i + 1] = ev.y;
                        pm = fmaxf(pm, fmaxf(fabsf(ev.x), fabsf(ev.y)));
                    }
                } else {
                    tc_fence_before();
                    if (h == 0) mbar_arrive(freeb + T);
                }
                EP_STAMP(2);
                if (h == 0) {
                    if (!TSM && l == 0 && (t0 > 0 || s > 0)) {  // the slot's scratch still holds the head partial sums of its previous tile
                        mbar_wait(hfree + T, (hfph >> T) & 1u);
                        hfph ^= 1u << T;
                        tc_fence_after();
                    }
                    if (wact) {  // park the first 16 activations until half 1 is done (only this thread reads them back)
                        tmem_st16f(stash, v);
                        tmem_wait_st();
                    }
                } else {
                    float u[16];
                    if (wact) {
                        tmem_ld16f(stash, u);
                        tmem_wait_ld();
#pragma unroll
                        for (int i = 0; i < 16; i += 2) pm = fmaxf(pm, fmaxf(fabsf(u[i]), fabsf(u[i + 1])));
                    }
                    if (l + 1 < NL) {
                        const float ncx = q2_quantise_store(c, T, wact, u, v, pm);
                        if (T) cx1 = ncx; else cx0 = ncx;
                    } else if (TSM) {
                        q2_heads_tsm(c, p, wact && c.r < nrows, u, v, smt.part, nrows);
                    } else {
                        q2_heads(c, p, T, wact, u, v);
                    }
                }
                EP_STAMP(3);
            }
        }
        if (FUSED) {
            // ---- tree phase: one thread per tree of the CTA
            const long long c0 = clock64();
            phase_sync(&phase_bar, pph);  // the post-processing warps have finished every row of this evaluation
            const long long c1 = clock64();
            if (TSM) {
                ds_phase(&s_dsctx, (s > 0 ? 1 : 0) | (s + 1 < n_evals ? 2 : 0));
            } else
#pragma unroll 1
            for (int i = tid; i < nrows; i += Q2_EPI_THREADS) {
                const int gr = row_begin + i;
                if constexpr (ENV::DISCRETE) {
                    d_step<ENV>(tp, tabs, gr, s > 0, s + 1 < n_evals);
                } else {
                    if (s == 0) c_root_insert(tp, gr);                // the add_pw_action(root) before the loop (mcts.py:673)
                    c_step<ENV>(tp, tabs, gr, s > 0, s + 1 < n_evals);  // backup of simulation s, descent + expansion of simulation s + 1
                }
            }
            phase_sync(&phase_bar, pph);
            cyc_sync += c1 - c0;
            cyc_tree += clock64() - c1;
#ifdef AZG_EVAL_PROF
            if (tid == 0) { s_dsprof[4] += (unsigned long long)(c1 - c0); s_dsprof[5] += (unsigned long long)(clock64() - c1); }
            ep_last = clock64();
#endif
        }
        }
        if (TSM) ds_writeback(tp, smt, nrows, row_begin, tid, Q2_EPI_THREADS);  // after the last phase boundary: the rows are final
        if (FUSED && tid == 0 && p.stats) {
            atomicAdd(p.stats + 0, (unsigned long long)(clock64() - cyc_begin));
            atomicAdd(p.stats + 1, (unsigned long long)cyc_tree);
            atomicAdd(p.stats + 2, (unsigned long long)cyc_sync);
            atomicAdd(p.stats + 4, 1ull);
#ifdef AZG_TREE_PROF
            if (TSM) for (int k = 0; k < 8; ++k) atomicAdd(p.stats + 8 + k, s_dsprof[k]);
#endif
#ifdef AZG_EVAL_PROF
            for (int k = 0; k < 8; ++k) atomicAdd(p.stats + 8 + k, s_dsprof[k]);
#endif
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tb), "n"(512) : "memory");
}

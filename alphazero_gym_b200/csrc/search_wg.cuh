// search_wg.cuh -- the WHOLE SEARCH in one persistent kernel, organised as FOUR INDEPENDENT WARPGROUPS per SM.
//
// Same arithmetic as qmlp2.cuh (AZG_FLAG_EVAL_Q8 contract: exact int8-sliced fixed-point products on tcgen05.mma kind::i8, bit-
// identical to the CPU oracle) and the same tree step (tree_continuous.cuh / tree_discrete.cuh); a different schedule.
//
// Why.  The two-phase kernel (qmlp2.cuh, FUSED) alternates an evaluation phase and a tree phase for the whole CTA.  ncu on it
// (profiles/r1i): the schedulers issue on 46 % of the cycles, no pipe is above 45 % busy, and instruction-count cuts in the
// epilogue barely move the time (-22 % instructions in the conversion block: -4 % time, profiles/README.md r2b).  Both phases are
// LATENCY bound: in the evaluation the 16 epilogue warps walk every step together (the four warps of a scheduler share a row
// group, meet at its named barrier and wait for the same tcgen05.ld), and the tree phase is a chain of dependent loads with 14
// warps and nothing else to issue.  The cure is independent instruction streams per scheduler, not fewer instructions.
//
// How.  A THREAD OWNS ONE TREE FOR THE WHOLE SEARCH -- its tree step AND its row of the network evaluation:
//   * warpgroup g (4 warps, 128 threads) owns tile g (g + 4, ... for larger batches) of at most 128 trees; thread r of the warpgroup
//     is TMEM lane r, i.e. row r of the tile's MMAs, and reads all 128 output columns of its row, 16 at a time;
//   * the row maximum (the scale of the next layer's fixed-point input) and the head dot products are thread-local: no named
//     barriers, no shared-memory exchange, no post-processing warps; leaf word, network input and evaluation results never
//     cross threads (the tree step that consumes an evaluation runs in the thread that produced it), so there are no
//     CTA-wide phase boundaries either;
//   * per simulation a warpgroup runs  evaluate(its tile) -> finish rows -> tree step (backup, select, expand)  at its own
//     pace.  The four warps of a scheduler belong to four different warpgroups: while one sits in the dependent-load chain
//     of its tree step the others issue evaluation arithmetic;
//   * the activations of a row wait for the row maximum in TMEM (128 stash columns per tile), so only TWO tiles fit the 512
//     TMEM columns at a time: two SLOTS (A-operand buffer + accumulator windows + stash), slot s shared by warpgroups s and
//     s + 2, which take turns (mbarrier `slotfree`); a warpgroup holds its slot only for layer 0 .. heads;
//   * every H x H layer is issued in eight N = 16 column STEPS into two alternating 48-column accumulator windows (PA | PB | PC),
//     so the MMAs of steps k + 1 and k + 2 run under the arithmetic of step k and the warps of a warpgroup meet only through
//     barriers that complete two steps ahead.  One MMA instruction costs ~46 cycles for any N <= 64 (tools/umma_n_probe.cu), so
//     the six digit products of a K step are issued as THREE instructions: the weight digit planes of a step are stored as 48
//     consecutive rows (hi | mid | lo), and xh x [wh | wm | wl] (N = 48) writes PA | PB | PC, xm x [wh | wm] (N = 32) adds into
//     PB | PC, xl x [wh] (N = 16) into PC; one issuing thread per slot.
// Synchronisation: mbarriers only (ready / full / accfree / slotfree per slot).
#pragma once
#include "qmlp2.cuh"

#define WG_THREADS 640          // 16 tree + evaluation warps (4 warpgroups) and the MMA warpgroup (two issuing threads)
#define WG_EPI_THREADS 512
#define WG_IDESC(N) ((2u << 4) | (1u << 7) | (1u << 10) | (((uint32_t)(N) >> 3) << 17) | ((128u >> 4) << 24))  // s8 x s8 -> s32, K-major, M = 128
#define WG_B_KCHUNK 6144        // weight digits of a layer: [k/16][step of 16 outputs][plane][16 rows][16 B]: bytes per 16-wide k chunk ...
#define WG_B_STEP 768           // ... and per step (3 planes x 16 rows x 16 B)
#define WG_WIN_COLS 48          // one accumulator window: PA | PB | PC, 16 columns each
#define WG_STASH_COL 96         // two accumulator windows in columns 0 .. 95 of the slot, then the stash of the row's 128 activations
#define WG_SLOT_COLS 224
#define WG_MAX_ROUNDS 4         // tiles per warpgroup and launch (engine.cu cuts larger batches into chunks)

__host__ __device__ inline size_t search_wg_smem_bytes(int NL, int qfl_count) {
    return (size_t)NL * 3 * QMLP_PLANE + 2 * 3 * QMLP_PLANE + (size_t)qfl_count * 4 + 1024 + Q2_TAB_BYTES;
}

__device__ __forceinline__ void umma_i8_wg(uint32_t tmem_d, uint32_t da_lo, uint32_t db_lo, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tmov.b64 da, {%1, %5};\n\tmov.b64 db, {%2, %5};\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], da, db, %3, p;\n\t}" ::"r"(tmem_d),
        "r"(da_lo), "r"(db_lo), "r"(idesc), "r"(accumulate), "r"(Q2_DESC_HI)
        : "memory");
}
__device__ __forceinline__ uint32_t wg_descb_lo(uint32_t saddr) { return ((saddr >> 4) & 0x3FFFu) | (((uint32_t)WG_B_KCHUNK >> 4) << 16); }

#ifndef WG_EPI_REGS
#define WG_EPI_REGS 104  // registers of a tree + evaluation thread / of an MMA-warpgroup thread after setmaxnreg (granularity 8).  112 / 24
#define WG_MMA_REGS 56   // measured worse: the issue loop spills at 24 (waiting for MMAs 6.6 % -> 15 %, 1142 -> 1035 M sims/s, r2z)
#endif

// mbarrier operations on a shared-memory ADDRESS (qmlp.cuh mbar_wait / qmlp2.cuh mbar_arrive take generic pointers)
__device__ __forceinline__ void mbar_arrive_s(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ bool mbar_try_wait_s(uint32_t bar, uint32_t parity, uint32_t ns) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity), "r"(ns) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait_s(uint32_t bar, uint32_t parity) {  // bounded like mbar_wait: a protocol error traps instead of hanging
    int spins = 0;
    while (!mbar_try_wait_s(bar, parity, 20000u)) {
        if (++spins > (1 << 22)) {
            printf("mbar_wait timeout: block %d thread %d barrier smem 0x%x parity %u\n", blockIdx.x, threadIdx.x, bar, parity);
            __trap();
        }
    }
}

// per-thread view of its slot
struct WgSlot {
    uint32_t tacc;      // TMEM address (lane quarter of this warp, first column of the slot)
    int8_t* sA;         // [3][QMLP_PLANE] A-operand digit planes of the slot
    uint32_t ready, full, accfree, slotfree;  // mbarriers as 32-bit shared addresses (half the registers of generic pointers, and no
                                              // conversion per use); full / accfree: [2] (one per accumulator window, + 8 bytes);
                                              // slotfree: [2] (one per warpgroup of the slot)
    uint32_t fullph;  // bit w: parity of the next wait on full[w]
    long long cyc_full;  // cycles spent waiting for MMAs (azg_fused_stats)
#ifdef AZG_EVAL_PROF
    long long cyc_k[3];  // ... of which at column step 0, step 1, steps 2..7
#endif
};

// scale of a row from its maximum, then the row's 128 stashed activations -> three digit planes in shared memory -> "ready"
__device__ __forceinline__ float wg_quantise_row(const WgSlot& sl, bool wact, int r, float pm) {
    float cx = 0.0f;
    if (wact) {
        const int e = q8_exponent(pm);
        const float sx = __uint_as_float((uint32_t)(276 - e) << 23);  // 2^(149-e)
        cx = __uint_as_float((uint32_t)(e - 22) << 23);               // 2^(e-149)
#pragma unroll 2
        for (int c = 0; c < 8; ++c) {
            float v[16];
            tmem_ld16f(sl.tacc + WG_STASH_COL + 16 * c, v);
            tmem_wait_ld();
            q8_store16(v, sx, sl.sA, c, r);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes of A -> visible to the tensor core
    }
    tc_fence_before();
    mbar_arrive_s(sl.ready);
    return cx;
}

// one evaluation of the warpgroup's tile (all 128 threads take part in the barrier protocol; `wact`: this warp has valid rows).
// Returns the value head and the raw policy-head outputs of this thread's row in out[].
template <int S, int ACT, int NL>
__device__ __forceinline__ void wg_evaluate(const MlpParams& p, WgSlot& sl, const float* fl, bool wact, bool valid, int gr, int r, float* out) {
    const float* W0 = fl;
    const float* b0 = fl + S * 128;
    const float2* cwb = reinterpret_cast<const float2*>(fl + S * 128 + 128);
    const float* Wh = fl + S * 128 + 128 + NL * 2 * 128;
    const float* bh = Wh + 128 * p.PO_PAD;
    // ---- layer 0 (S -> H) in FP32 FMA, 16 outputs at a time, activations parked in the stash
    float pm = 0.0f;
    if (wact) {
        float x[S];
#pragma unroll
        for (int s = 0; s < S; ++s) x[s] = 0.0f;
        if (valid) {
            if constexpr (S > 4) {  // Acrobot: 6 inputs in two float4 per leaf
                const float4 v = *reinterpret_cast<const float4*>(p.X + (size_t)gr * 8), w = *reinterpret_cast<const float4*>(p.X + (size_t)gr * 8 + 4);
                x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w; x[4] = w.x; x[5] = w.y;
            } else {
                const float4 v = *reinterpret_cast<const float4*>(p.X + (size_t)gr * 4);
                x[0] = v.x; x[1] = v.y;
                if constexpr (S > 2) x[2] = v.z;
                if (S > 3) x[S - 1] = v.w;
            }
        }
#pragma unroll 1
        for (int c = 0; c < 8; ++c) {
            float a[16];
#pragma unroll
            for (int i = 0; i < 16; i += 2) {
                const int j = c * 16 + i;
                float2 acc = *reinterpret_cast<const float2*>(b0 + j);
#pragma unroll
                for (int s = 0; s < S; ++s) acc = __ffma2_rn(make_float2(x[s], x[s]), *reinterpret_cast<const float2*>(W0 + s * 128 + j), acc);
                const float2 e = mlp_act2<ACT>(acc);
                a[i] = e.x; a[i + 1] = e.y;
                pm = fmaxf(pm, fmaxf(fabsf(e.x), fabsf(e.y)));
            }
            tmem_st16f(sl.tacc + WG_STASH_COL + 16 * c, a);
        }
        tmem_wait_st();
    }
    float cx = wg_quantise_row(sl, wact, r, pm);
    // ---- hidden layers: eight N = 16 steps per layer, accumulator windows alternate
#pragma unroll 1
    for (int l = 0; l < NL; ++l) {
        pm = 0.0f;
#pragma unroll 1
        for (int k = 0; k < 8; ++k) {
            const int w = k & 1;
            const long long f0 = clock64();
            mbar_wait_s(sl.full + 8u * w, (sl.fullph >> w) & 1u);
            sl.fullph ^= 1u << w;
            tc_fence_after();
            sl.cyc_full += clock64() - f0;
#ifdef AZG_EVAL_PROF
            sl.cyc_k[k < 2 ? k : 2] += clock64() - f0;
#endif
            if (wact) {
                const uint32_t ta = sl.tacc + w * WG_WIN_COLS;
                int32_t pa[16], pb[16], pc[16];
                tmem_ld16(ta, pa);
                tmem_ld16(ta + 16, pb);
                tmem_ld16(ta + 32, pc);
                tmem_wait_ld();
                tc_fence_before();
                if (k < 6) mbar_arrive_s(sl.accfree + 8u * w);  // the window may be overwritten by the MMAs of step k + 2
                const float2* cb = cwb + l * 128 + 16 * k;
                float v[16];
#pragma unroll
                for (int i = 0; i < 16; i += 2) {
                    const float4 sb = *reinterpret_cast<const float4*>(cb + i);  // (cw, bias) of outputs i, i + 1
                    // fma(PA, 256, PB) of the contract = the correctly rounded integer PA * 256 + PB (see qmlp2.cuh)
                    float u0 = __int2float_rn(pa[i] * 256 + pb[i]);
                    float u1 = __int2float_rn(pa[i + 1] * 256 + pb[i + 1]);
                    u0 = __fmaf_rn(u0, 256.0f, q8_i2f_23(pc[i]));
                    u1 = __fmaf_rn(u1, 256.0f, q8_i2f_23(pc[i + 1]));
                    const float2 y = make_float2(__fmaf_rn(u0, __fmul_rn(cx, sb.x), sb.y), __fmaf_rn(u1, __fmul_rn(cx, sb.z), sb.w));
                    const float2 ev = mlp_act2<ACT>(y);
                    v[i] = ev.x; v[i + 1] = ev.y;
                    pm = fmaxf(pm, fmaxf(fabsf(ev.x), fabsf(ev.y)));
                }
                tmem_st16f(sl.tacc + WG_STASH_COL + 16 * k, v);
            } else {
                tc_fence_before();
                if (k < 6) mbar_arrive_s(sl.accfree + 8u * w);
            }
        }
        if (wact) tmem_wait_st();
        if (l + 1 < NL) cx = wg_quantise_row(sl, wact, r, pm);
    }
    // ---- heads: the four 32-activation FMA chains of the contract (column quarters), summed as ((q0 + q1) + (q2 + q3)) + bias
    if (wact) {
#pragma unroll 1
        for (int c4 = 0; c4 < p.PO_PAD / 4; ++c4) {
            float2 lo[4], hi[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                lo[q] = make_float2(0.0f, 0.0f);
                hi[q] = make_float2(0.0f, 0.0f);
#pragma unroll
                for (int hc = 0; hc < 2; ++hc) {
                    float a[16];
                    tmem_ld16f(sl.tacc + WG_STASH_COL + 32 * q + 16 * hc, a);
                    tmem_wait_ld();
                    const float* wp = Wh + (32 * q + 16 * hc) * p.PO_PAD + c4 * 4;
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        const float4 w4 = *reinterpret_cast<const float4*>(wp + i * p.PO_PAD);
                        const float2 av = make_float2(a[i], a[i]);
                        lo[q] = __ffma2_rn(av, make_float2(w4.x, w4.y), lo[q]);
                        hi[q] = __ffma2_rn(av, make_float2(w4.z, w4.w), hi[q]);
                    }
                }
            }
            const float s0 = __fadd_rn(__fadd_rn(__fadd_rn(lo[0].x, lo[1].x), __fadd_rn(lo[2].x, lo[3].x)), bh[c4 * 4 + 0]);
            const float s1 = __fadd_rn(__fadd_rn(__fadd_rn(lo[0].y, lo[1].y), __fadd_rn(lo[2].y, lo[3].y)), bh[c4 * 4 + 1]);
            const float s2 = __fadd_rn(__fadd_rn(__fadd_rn(hi[0].x, hi[1].x), __fadd_rn(hi[2].x, hi[3].x)), bh[c4 * 4 + 2]);
            const float s3 = __fadd_rn(__fadd_rn(__fadd_rn(hi[0].y, hi[1].y), __fadd_rn(hi[2].y, hi[3].y)), bh[c4 * 4 + 3]);
#pragma unroll  // static indices: out[] stays in registers
            for (int g4 = 0; g4 < Q2_MAX_PO / 4; ++g4)
                if (g4 == c4) { out[4 * g4] = s0; out[4 * g4 + 1] = s1; out[4 * g4 + 2] = s2; out[4 * g4 + 3] = s3; }
        }
    }
    tc_fence_before();
}

// ENV (env.cuh): CartPole = the discrete tree, Pendulum | MountainCarContinuous = the continuous tree stepping that env
template <class ENV, int ACT, int NL>
__global__ void __launch_bounds__(WG_THREADS, 1)
k_search_wg(const MlpParams p, const TreeParams tp, const int n_sims, const int chunk_begin, const int chunk_end) {
    constexpr int S = ENV::S;
    extern __shared__ __align__(1024) uint8_t wsm_raw[];
    __shared__ __align__(8) uint64_t wbar, ready[2], full[2][2], accfree[2][2], slotfree[2][2];
    __shared__ uint32_t tmem_base_s;
    uint8_t* qsm = wsm_raw + ((1024u - (smem_u32(wsm_raw) & 1023u)) & 1023u);  // offset on the shared pointer (keeps the address space)
    int8_t* sB = reinterpret_cast<int8_t*>(qsm);                    // [NL][3][8][128][16], rows in natural order
    int8_t* sA = sB + (size_t)NL * 3 * QMLP_PLANE;                  // [2 slots][3][8][128][16]
    float* fl = reinterpret_cast<float*>(sA + 2 * 3 * QMLP_PLANE);  // W0t[S][H], b0[H], NL x (cw, bias)[H], Wh[H][PO_PAD], bh[PO_PAD]
    double* s_rcp = reinterpret_cast<double*>(fl + p.qfl_count);
    double* s_sq = s_rcp + FUSED_TAB + 1;
    int32_t* s_pw = reinterpret_cast<int32_t*>(s_sq + FUSED_TAB + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int per = (chunk_end - chunk_begin + gridDim.x - 1) / gridDim.x;
    const int row_begin = chunk_begin + blockIdx.x * per;
    const int row_end = min(row_begin + per, chunk_end);
    if (row_begin >= row_end) return;
    const int nrows = row_end - row_begin;
    // tiles: 4 per round (one per warpgroup); full warps first, small batches spread over the four warpgroups
    const int rounds = (nrows + 511) / 512;
    const int ntiles_max = 4 * rounds;
    int th = (nrows + ntiles_max - 1) / ntiles_max;
    if (th > 32) th = (th + 31) & ~31;
    const int ntiles = (nrows + th - 1) / th;
    const int n_evals = n_sims + 1;  // evaluations per tree: the root + one per simulation

    if (tid == 0) {
        mbar_init(&wbar, 1);
        for (int s = 0; s < 2; ++s) {
            mbar_init(&ready[s], 128);
            mbar_init(&slotfree[s][0], 128);
            mbar_init(&slotfree[s][1], 128);
            for (int w = 0; w < 2; ++w) {
                mbar_init(&full[s][w], 1);
                mbar_init(&accfree[s][w], 128);
            }
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
#ifdef AZG_WG_DEBUG
    if (tid == 0 && blockIdx.x == 0)
        printf("wg: wbar 0x%x ready 0x%x full 0x%x accfree 0x%x slotfree 0x%x tmem 0x%x nrows %d th %d ntiles %d rounds %d\n", smem_u32(&wbar), smem_u32(ready),
               smem_u32(&full[0][0]), smem_u32(&accfree[0][0]), smem_u32(&slotfree[0][0]), tb, nrows, th, ntiles, rounds);
#endif
    if (tid == 0) {
        const uint32_t bytesB = (uint32_t)NL * 3 * QMLP_PLANE, bytesF = (uint32_t)p.qfl_count * 4u;
        mbar_expect_tx(&wbar, bytesB + bytesF);
        for (uint32_t o = 0; o < bytesB; o += 32768u) bulk_g2s(sB + o, p.qdigits_nat + o, min(32768u, bytesB - o), &wbar);
        bulk_g2s(fl, p.qfl, bytesF, &wbar);
    }
    for (int i = tid; i <= FUSED_TAB; i += blockDim.x) {
        s_rcp[i] = tp.rcp_tab[i];
        s_sq[i] = tp.sqrt_tab[i];
        s_pw[i] = (tp.pw_table && i < p.R) ? tp.pw_table[i] : 0;  // continuous only; the table has max_rollouts + 2 = R entries
    }
    __syncthreads();
    mbar_wait(&wbar, 0);

    if (warp >= 16) {
        // ---- MMA warpgroup: gives its registers away; warps 16 and 17 issue for slot 0 and slot 1.  The whole warp runs the loop, so
        // that descriptors and window addresses are warp-uniform (uniform registers), and one elected lane issues the tcgen05
        // instructions (qmlp2.cuh elect_one: with the loop under `lane == 0` every UTCIMMA carried ~12 instructions of R2UR traffic)
        // (56 registers: with the 24 of qmlp2.cuh the issue loop below spills its descriptors, and a local-memory reload in front of
        // every tcgen05.mma -- this kernel has almost no L1 -- made an MMA cost ~290 cycles instead of ~46, profiles/README.md r2b)
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(WG_MMA_REGS));
        if (warp < 18) {
            const int slot = warp - 16;
            uint32_t rph = 0, aph = 0;  // parity of the next wait on ready[slot]; bit w: on accfree[slot][w]
            const uint32_t aH = q2_desc_lo(smem_u32(sA) + (uint32_t)slot * 3 * QMLP_PLANE), aM = aH + 1024, aL = aH + 2048;
#pragma unroll 1
            for (int s = 0; s < n_evals; ++s)
#pragma unroll 1
            for (int rd = 0; rd < rounds; ++rd)
#pragma unroll 1
            for (int half = 0; half < 2; ++half) {
                if (4 * rd + slot + 2 * half >= ntiles) continue;  // the warpgroup makes an empty use of the slot
#pragma unroll 1
                for (int l = 0; l < NL; ++l) {
#pragma unroll 1
                    for (int k = 0; k < 8; ++k) {
                        const int w = k & 1;
                        if (k == 0) { mbar_wait(&ready[slot], rph); rph ^= 1u; }
                        else if (k >= 2) { mbar_wait(&accfree[slot][w], (aph >> w) & 1u); aph ^= 1u << w; }
                        tc_fence_after();
                        // A: +1024 per digit plane (16 KB), +256 per K step of 32 (two k chunks of 2 KB).  B: the 48 rows hi | mid | lo of
                        // step k; +768 per K step (two k chunks of 6 KB)
                        const uint32_t bq = wg_descb_lo(smem_u32(sB) + (uint32_t)l * 3 * QMLP_PLANE + (uint32_t)k * WG_B_STEP);
                        const uint32_t acc = tb + slot * WG_SLOT_COLS + w * WG_WIN_COLS;
                        if (elect_one()) {
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) {
                            umma_i8_wg(acc, aH + kk * 256, bq + kk * 768, WG_IDESC(48), kk > 0);   // PA | PB | PC  = / += xh x [wh | wm | wl]
                            umma_i8_wg(acc + 16, aM + kk * 256, bq + kk * 768, WG_IDESC(32), 1);    //      PB | PC += xm x [wh | wm]
                            umma_i8_wg(acc + 32, aL + kk * 256, bq + kk * 768, WG_IDESC(16), 1);    //           PC += xl x [wh]
                        }
                        umma_commit(&full[slot][w]);
                        }
                        __syncwarp();
                    }
                }
            }
        }
    } else {
        // ---- tree + evaluation warpgroups
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(WG_EPI_REGS));  // 512 x 104 + 128 x 56 = 60416 <= 640 x 96, the CTA's pool at launch (engine.cu checks it)
        const int g = warp >> 2, slot = g & 1, half = g >> 1;
        const int r = (warp & 3) * 32 + lane;  // row of the tile = TMEM lane
        WgSlot sl;
        sl.tacc = tb + ((uint32_t)((warp & 3) * 32) << 16) + slot * WG_SLOT_COLS;
        sl.sA = sA + (size_t)slot * 3 * QMLP_PLANE;
        sl.ready = smem_u32(&ready[slot]); sl.full = smem_u32(full[slot]); sl.accfree = smem_u32(accfree[slot]); sl.slotfree = smem_u32(slotfree[slot]);
        sl.fullph = 0;
        sl.cyc_full = 0;
#ifdef AZG_EVAL_PROF
        sl.cyc_k[0] = sl.cyc_k[1] = sl.cyc_k[2] = 0;
#endif
        bool first_use = true;
        uint32_t useph = 0;  // parity of the next wait on the other warpgroup's release barrier
        const Tabs tabs = {s_pw, s_rcp, s_sq, FUSED_TAB};
        long long cyc_tree = 0, cyc_slot = 0;
        const long long cyc_begin = clock64();
        uint32_t nev = 0;
        int ev_row = 0;
        // initialize_search for every tree of the warpgroup
        for (int rd = 0; rd < rounds; ++rd) {
            const int tile = 4 * rd + g, row0 = row_begin + tile * th;
            if (tile < ntiles && row0 + r < min(row0 + th, row_end)) {
                if constexpr (ENV::DISCRETE) d_init<ENV>(tp, row0 + r);
                else c_init<ENV>(tp, row0 + r);
            }
        }
#pragma unroll 1
        for (int s = 0; s < n_evals; ++s) {
#pragma unroll 1
        for (int rd = 0; rd < rounds; ++rd) {
            const int tile = 4 * rd + g;
            const bool tvalid = tile < ntiles;
            const int row0 = row_begin + tile * th;
            const int nv = tvalid ? max(0, min(th, row_end - row0)) : 0;
            const int gr = row0 + r;
            const bool valid = r < nv, wact = (warp & 3) * 32 < nv;
            // ---- take the slot (the other warpgroup of the slot has released its use)
            const long long c0 = clock64();
            // uses of a slot alternate between its two warpgroups; each warpgroup releases on its OWN mbarrier (slotfree[slot][half])
            // and waits on the other's, so every thread waits for consecutive phases of a barrier (a parity wait tells only two
            // consecutive phases apart: one barrier for both warpgroups lets a fast thread slip a whole use ahead)
            if (half == 1 || !first_use) {
                mbar_wait_s(sl.slotfree + 8u * (half ^ 1), useph);
                useph ^= 1u;
            }
            first_use = false;
            tc_fence_after();
            const long long c1 = clock64();
            float out[Q2_MAX_PO];
#pragma unroll
            for (int i = 0; i < Q2_MAX_PO; ++i) out[i] = 0.0f;
            if (tvalid) wg_evaluate<S, ACT, NL>(p, sl, fl, wact, valid, gr, r, out);
            mbar_arrive_s(sl.slotfree + 8u * half);  // TMEM and the A buffer of the slot are free again
            const long long c2 = clock64();
            // ---- finish the row, then the tree step of this thread's tree
            if (valid) {
                int leafw;
                double lr = 0.0;
                if (p.variant == 1) {
                    const uint4 k0 = p.ctl[gr], k1 = p.ctl[(size_t)p.BS + gr];
                    leafw = (int)k0.z;
                    lr = __hiloint2double((int)k1.w, (int)k1.z);
                } else {
                    leafw = p.leaf[gr];
                }
                if (leafw & LEAF_EVAL) {
                    mlp_finish_row<env::row3<ENV>()>(p, gr, leafw, lr, out[0], out + 1);
                    ++nev;
                    ev_row = gr;
                }
                if constexpr (ENV::DISCRETE) {
                    d_step<ENV>(tp, tabs, gr, s > 0, s + 1 < n_evals);
                } else {
                    if (s == 0) c_root_insert(tp, gr);             // the add_pw_action(root) before the loop (mcts.py:673)
                    c_step<ENV>(tp, tabs, gr, s > 0, s + 1 < n_evals);  // backup of simulation s, descent + expansion of simulation s + 1
                }
            }
            cyc_slot += c1 - c0;
            cyc_tree += clock64() - c2;
        }
        }
        if (nev) p.evals[ev_row] += nev;  // only the total over trees is reported (azg_get_counters)
        if ((warp & 3) == 0 && lane == 0 && p.stats) {
            atomicAdd(p.stats + 0, (unsigned long long)(clock64() - cyc_begin));
            atomicAdd(p.stats + 1, (unsigned long long)cyc_tree);
            atomicAdd(p.stats + 2, (unsigned long long)cyc_slot);
            atomicAdd(p.stats + 3, (unsigned long long)sl.cyc_full);
#ifdef AZG_EVAL_PROF
            for (int k = 0; k < 3; ++k) atomicAdd(p.stats + 8 + k, (unsigned long long)sl.cyc_k[k]);
#endif
            atomicAdd(p.stats + 4, 1ull);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tb), "n"(512) : "memory");
}

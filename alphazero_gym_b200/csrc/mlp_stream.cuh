// mlp_stream.cuh -- batched FP32 leaf evaluation for the hidden widths whose weights do not fit in shared memory.
//
// k_mlp (mlp.cuh) stages the whole network in shared memory once per CTA, which stops at hidden = 128: one 256 x 256 f32 layer is
// 256 KB, more than the 227 KB a block can have.  k_mlp_stream serves every other multiple of 32 up to 256 with the same numerical
// contract (AZO_EVAL_FP32 of the oracle, bit for bit): every layer output is acc = bias; acc = fma(w[j][k], x[k], acc) for k ascending,
// the activations are mlp_act2<ACT>, the heads put value_head in column 0 and dist_head in columns 1..P, and every row is finished by
// mlp_finish_row.  The width is a run-time value (MlpStreamPlan); only the input width S and the activation are template arguments.
//
// Structure (one persistent CTA per SM, or per 64 rows in a thin batch; 32 x NB x RB threads, NB = H / 32 column blocks, RB = 64-row
// blocks per pass):
//   * layer 0 and the heads are small and stay resident in shared memory (one TMA bulk copy each at the start);
//   * the CTA owns a contiguous share of the rows and evaluates it in passes of RP = 64 x RB rows, activations k-major [H][RP];
//   * each hidden layer's Wt[H][H] streams through a ring of MLPS_STAGES slices of MLPS_KS k-rows (cp.async.bulk into a stage whose
//     `full` mbarrier counts the bytes; every warp arrives on the stage's `empty` mbarrier once it has read the slice).  The slices of
//     all layers and passes form one sequence; thread 0 refills the stage of slice g - 2 with slice g + MLPS_STAGES - 2 when it starts
//     slice g, so two slices are in flight ahead of the slowest warp and thread 0 seldom waits;
//   * a warp owns a 64-row x 32-column tile (two of k_mlp's 32 x 32 tiles sharing their weight operands): per k each thread reads two
//     float4 of activations and two float4 of weights for 32 packed FFMA2 (k_mlp: one and two for 16);
//   * warps whose 64-row block lies past the rows of a ragged last pass skip the arithmetic but still wait and arrive on every slice.
// Bound: FP32 FMA issue, plus the phases that run between the hidden layers with every warp of the CTA in them (layer 0, the heads and
// the post-processing).  Weight traffic from L2: (passes) x (L - 1)(H^2 + H) x 4 bytes per evaluation.
#pragma once
#include "mlp.cuh"

#define MLPS_MAX_THREADS 512  // 16 warps: NB x RB <= 16
#define MLPS_KS 8             // k-rows of Wt per streamed slice
#define MLPS_STAGES 4         // slices in the ring

// the shape of one engine's network and its pass size, computed once by azg_create (engine.cu)
struct MlpStreamPlan {
    int32_t H;          // hidden width: a multiple of 32, at most 256
    int32_t NB, RB;     // 32-column blocks (H / 32) and 64-row blocks per pass; the CTA has NB x RB warps
    int32_t RP;         // rows per pass (64 x RB)
    int32_t w0_floats;  // layer 0 in wpack: W0t[S][H] + b0[H]
    int32_t head_off;   // heads in wpack: Wh[H][PO_PAD] + bh[PO_PAD], from this float on
};

// shared memory of k_mlp_stream (the layout at the top of the kernel; all of it dynamic, mbarriers included), bytes
__host__ __device__ inline size_t mlp_stream_smem_bytes(int H, int S, int PO_PAD, int RP) {
    const size_t floats = (size_t)MLPS_STAGES * MLPS_KS * H + (size_t)S * H + H + (size_t)H * PO_PAD + PO_PAD + (size_t)H * RP +
                          (size_t)PO_PAD * RP + (size_t)S * RP + RP;
    return floats * sizeof(float) + (size_t)RP * sizeof(double) + (2 * MLPS_STAGES + 1) * sizeof(uint64_t);
}

template <int S, int ACT>
__global__ void __launch_bounds__(MLPS_MAX_THREADS, 1) k_mlp_stream(const MlpParams p, const MlpStreamPlan sp) {
    extern __shared__ __align__(128) float smem[];
    const int H = sp.H, RP = sp.RP, PO = p.PO_PAD;
    const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = nthr >> 5;
    const int slice = MLPS_KS * H;  // floats per slice
    float* ring = smem;                                    // [MLPS_STAGES][MLPS_KS][H]
    float* w0 = ring + MLPS_STAGES * slice;                // W0t[S][H], b0[H]
    float* wh = w0 + sp.w0_floats;                         // Wh[H][PO], bh[PO]
    float* act = wh + H * PO + PO;                         // [H][RP] activations, k-major
    float* outs = act + H * RP;                            // [PO][RP] raw head outputs
    float* xs = outs + PO * RP;                            // [S][RP] inputs
    int* rinfo = reinterpret_cast<int*>(xs + S * RP);      // [RP] leaf word, LEAF_EVAL set where the row is evaluated
    double* rlr = reinterpret_cast<double*>(rinfo + RP);   // [RP] continuous: leafR before this evaluation
    uint64_t* full = reinterpret_cast<uint64_t*>(rlr + RP);  // [MLPS_STAGES] a slice has landed in the stage
    uint64_t* empty = full + MLPS_STAGES;                    // [MLPS_STAGES] every warp has read the stage's slice
    uint64_t& wbar = empty[MLPS_STAGES];                     // layer 0 and the heads have landed

    // this CTA's rows: an even split of n
    const int lo = (int)((long long)blockIdx.x * p.n / gridDim.x);
    const int hi = (int)((long long)(blockIdx.x + 1) * p.n / gridDim.x);
    if (lo >= hi) return;
    const int passes = (hi - lo + RP - 1) / RP;
    const int nks = H / MLPS_KS;
    const int total = passes * (p.L - 1) * nks;  // slices this CTA streams

    // slice g of the sequence: layer 1 + (g / nks) % (L - 1), k-rows [(g % nks) * MLPS_KS, + MLPS_KS)
    auto issue = [&](int g) {
        const int s = g % MLPS_STAGES;
        if (g >= MLPS_STAGES)  // the stage's previous slice (g - MLPS_STAGES) has been read by every warp
            while (!mbar_try_wait(&empty[s], (uint32_t)(g / MLPS_STAGES - 1) & 1u)) {}
        const int l = 1 + (g / nks) % (p.L - 1);
        const float* src = p.wpack + sp.w0_floats + (size_t)(l - 1) * ((size_t)H * H + H) + (size_t)(g % nks) * slice;
        mbar_expect_tx(&full[s], (uint32_t)slice * 4u);
        bulk_g2s(ring + s * slice, src, (uint32_t)slice * 4u, &full[s]);
    };

    if (tid == 0) {
        for (int s = 0; s < MLPS_STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], nwarps);
        }
        mbar_init(&wbar, 1);
    }
    __syncthreads();
    if (tid == 0) {
        const uint32_t b0 = (uint32_t)sp.w0_floats * 4u, bh = (uint32_t)(H * PO + PO) * 4u;
        mbar_expect_tx(&wbar, b0 + bh);
        bulk_g2s(w0, p.wpack, b0, &wbar);
        bulk_g2s(wh, p.wpack + sp.head_off, bh, &wbar);
        for (int g = 0; g < MLPS_STAGES && g < total; ++g) issue(g);
    }
    while (!mbar_try_wait(&wbar, 0)) {}

    // hidden-layer tile of this warp: rows rb*64 + [0, 64), columns cb*32 + [0, 32); per thread rows r0 + {0..3} and r0 + 32 + {0..3},
    // columns c0 + {0..7}
    const int cb = warp % sp.NB, rb = warp / sp.NB;
    const int r0 = rb * 64 + (lane & 7) * 4, c0 = cb * 32 + (lane >> 3) * 8;
    int g = 0;  // next slice of the sequence

    for (int pass = 0; pass < passes; ++pass) {
        const int row0 = lo + pass * RP;
        const int nrows = min(RP, hi - row0);
        const int rows64 = (nrows + 63) & ~63;  // rows the hidden layers compute
        // ---- rows: leaf word, leafR and input (zero where the row is not evaluated, as in k_mlp)
        for (int r = tid; r < rows64; r += nthr) {
            const int gr = row0 + r;
            int leafw = 0;
            double lr = 0.0;
            bool need = r < nrows;
            if (need && p.mode == 0) {
                if (p.variant == 1) {  // continuous: leaf word and leafR share the first 32 B of the control block
                    const uint4 c0v = p.ctl[gr], c1v = p.ctl[(size_t)p.BS + gr];
                    leafw = (int)c0v.z;
                    lr = __hiloint2double((int)c1v.w, (int)c1v.z);
                } else {
                    leafw = p.leaf[gr];
                }
                need = (leafw & LEAF_EVAL) != 0;
            }
            rinfo[r] = need ? (leafw | LEAF_EVAL) : 0;
            rlr[r] = lr;
#pragma unroll
            for (int s = 0; s < S; ++s) xs[s * RP + r] = need ? p.X[(size_t)gr * p.xstride + s] : 0.0f;
        }
        __syncthreads();
        // ---- layer 0: S -> H, one (row, column pair) per item
        for (int i = tid; i < rows64 * (H / 2); i += nthr) {
            const int r = i % rows64, j = 2 * (i / rows64);
            float2 acc = *reinterpret_cast<const float2*>(w0 + S * H + j);
#pragma unroll
            for (int s = 0; s < S; ++s) {
                const float x = xs[s * RP + r];
                acc = __ffma2_rn(make_float2(x, x), *reinterpret_cast<const float2*>(w0 + s * H + j), acc);
            }
            const float2 e = mlp_act2<ACT>(acc);
            act[j * RP + r] = e.x;
            act[(j + 1) * RP + r] = e.y;
        }
        __syncthreads();
        // ---- hidden layers, Wt streamed through the ring
        const bool busy = rb * 64 < nrows;
        for (int l = 1; l < p.L; ++l) {
            const float* bias = p.wpack + sp.w0_floats + (size_t)(l - 1) * ((size_t)H * H + H) + (size_t)H * H;
            float2 acc[2][4][4];  // [row group][row][column pair]
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const float2 bc = __ldg(reinterpret_cast<const float2*>(bias + c0 + 2 * c));
#pragma unroll
                for (int h = 0; h < 2; ++h)
#pragma unroll
                    for (int r = 0; r < 4; ++r) acc[h][r][c] = bc;
            }
            for (int js = 0; js < nks; ++js, ++g) {
                if (tid == 0 && g >= 2 && g + MLPS_STAGES - 2 < total) issue(g + MLPS_STAGES - 2);
                const int s = g % MLPS_STAGES;
                while (!mbar_try_wait(&full[s], (uint32_t)(g / MLPS_STAGES) & 1u)) {}
                if (busy) {
                    const float* wk = ring + s * slice + c0;
                    const float* ak = act + js * MLPS_KS * RP + r0;
                    float4 a0 = *reinterpret_cast<const float4*>(ak), a1 = *reinterpret_cast<const float4*>(ak + 32);
                    float4 w0v = *reinterpret_cast<const float4*>(wk), w1v = *reinterpret_cast<const float4*>(wk + 4);
#pragma unroll 1
                    for (int k = 0; k < MLPS_KS; ++k) {
                        const int kn = k + 1 < MLPS_KS ? k + 1 : k;  // the last iteration re-reads row k (discarded)
                        const float4 na0 = *reinterpret_cast<const float4*>(ak + kn * RP);
                        const float4 na1 = *reinterpret_cast<const float4*>(ak + kn * RP + 32);
                        const float4 nw0 = *reinterpret_cast<const float4*>(wk + kn * H);
                        const float4 nw1 = *reinterpret_cast<const float4*>(wk + kn * H + 4);
                        const float ar[2][4] = {{a0.x, a0.y, a0.z, a0.w}, {a1.x, a1.y, a1.z, a1.w}};
                        const float2 wp[4] = {make_float2(w0v.x, w0v.y), make_float2(w0v.z, w0v.w), make_float2(w1v.x, w1v.y),
                                              make_float2(w1v.z, w1v.w)};
#pragma unroll
                        for (int h = 0; h < 2; ++h)
#pragma unroll
                            for (int r = 0; r < 4; ++r) {
                                const float2 av = make_float2(ar[h][r], ar[h][r]);
#pragma unroll
                                for (int c = 0; c < 4; ++c) acc[h][r][c] = __ffma2_rn(av, wp[c], acc[h][r][c]);
                            }
                        a0 = na0; a1 = na1; w0v = nw0; w1v = nw1;
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[s]);
            }
            __syncthreads();  // every warp has finished reading this layer's input
            if (busy) {
                // the raw sums first, then the activation over this thread's own outputs: the 64 accumulators are dead before the
                // activation's temporaries are live (mlp_act2 is elementwise, so any pairing gives the same bits)
#pragma unroll
                for (int h = 0; h < 2; ++h)
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        float* d0 = act + (c0 + 2 * c) * RP + r0 + 32 * h;
                        *reinterpret_cast<float4*>(d0) = make_float4(acc[h][0][c].x, acc[h][1][c].x, acc[h][2][c].x, acc[h][3][c].x);
                        *reinterpret_cast<float4*>(d0 + RP) = make_float4(acc[h][0][c].y, acc[h][1][c].y, acc[h][2][c].y, acc[h][3][c].y);
                    }
                __syncwarp();
#pragma unroll
                for (int h = 0; h < 2; ++h)
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        float4* d = reinterpret_cast<float4*>(act + (c0 + c) * RP + r0 + 32 * h);
                        const float4 v = *d;
                        const float2 e0 = mlp_act2<ACT>(make_float2(v.x, v.y)), e1 = mlp_act2<ACT>(make_float2(v.z, v.w));
                        *d = make_float4(e0.x, e0.y, e1.x, e1.y);
                    }
            }
            __syncthreads();
        }
        // ---- heads: column 0 = value_head, columns 1..P = dist_head; one (row, 4 columns) per item, k_mlp's operation order
        for (int i = tid; i < nrows * (PO / 4); i += nthr) {
            const int r = i % nrows, c = i / nrows;
            const float4 b4 = *reinterpret_cast<const float4*>(wh + H * PO + c * 4);
            float2 lo2 = make_float2(b4.x, b4.y), hi2 = make_float2(b4.z, b4.w);
#pragma unroll 8
            for (int k = 0; k < H; ++k) {
                const float a = act[k * RP + r];
                const float4 w4 = *reinterpret_cast<const float4*>(wh + k * PO + c * 4);
                const float2 av = make_float2(a, a);
                lo2 = __ffma2_rn(av, make_float2(w4.x, w4.y), lo2);
                hi2 = __ffma2_rn(av, make_float2(w4.z, w4.w), hi2);
            }
            outs[(c * 4 + 0) * RP + r] = lo2.x;
            outs[(c * 4 + 1) * RP + r] = lo2.y;
            outs[(c * 4 + 2) * RP + r] = hi2.x;
            outs[(c * 4 + 3) * RP + r] = hi2.y;
        }
        __syncthreads();
        // ---- post-processing + write-back, one thread per row
        for (int r = tid; r < nrows; r += nthr) {
            const int leafw = rinfo[r];
            if (!(leafw & LEAF_EVAL)) continue;
            float raw[3 * AZG_MAX_K];
            for (int i = 0; i < p.P; ++i) raw[i] = outs[(1 + i) * RP + r];
            mlp_finish_row<true>(p, row0 + r, leafw, rlr[r], outs[r], raw);
            if (p.mode == 0) p.evals[row0 + r] += 1;
        }
        __syncthreads();  // the next pass rewrites the row tables
    }
}

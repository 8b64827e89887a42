// primitives_probe.cu -- elementwise kernels around the engine's numeric and random primitives, for tests/test_primitives_gpu.py.
//
// The engine headers are included unchanged, and the file is compiled with the engine's own nvcc flags
// (alphazero_gym_b200/build.py NVCC_FLAGS, -fmad=false on sm_100a), so every probe runs exactly the code the kernels run.
// Each launcher takes device pointers, an element count and a stream.  Where a sweep covers every f32 bit pattern, the
// kernel makes its input from the element index (bits = mul * (base + i) + add), so nothing has to be copied in.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../alphazero_gym_b200/csrc/common.cuh"
#include "../alphazero_gym_b200/csrc/detmath.cuh"
#include "../alphazero_gym_b200/csrc/env.cuh"
#include "../alphazero_gym_b200/csrc/mlp.cuh"
#include "../alphazero_gym_b200/csrc/tree_discrete.cuh"

#define GRID(n) (unsigned)(((n) + 255) / 256 < 65536 ? ((n) + 255) / 256 : 65536), 256
#define FOR_EACH(i, n) for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < (n); i += (int64_t)gridDim.x * blockDim.x)

__device__ __forceinline__ float gen_f32(const uint32_t* in, uint32_t mul, uint32_t add, uint64_t base, int64_t i) {
    return __uint_as_float(in ? in[i] : mul * (uint32_t)(base + (uint64_t)i) + add);
}

// fn: 0 det::expf_, 1 det::expm1f_, 2 det::tanhf_, 16 + ACT mlp_act<ACT>
__global__ void k_f32(int fn, const uint32_t* in, uint32_t mul, uint32_t add, uint64_t base, float* out, int64_t n) {
    FOR_EACH(i, n) {
        const float x = gen_f32(in, mul, add, base, i);
        float y;
        switch (fn) {
            case 0: y = det::expf_(x); break;
            case 1: y = det::expm1f_(x); break;
            case 2: y = det::tanhf_(x); break;
            case 16: y = mlp_act<0>(x); break;
            case 17: y = mlp_act<1>(x); break;
            case 18: y = mlp_act<2>(x); break;
            case 19: y = mlp_act<3>(x); break;
            case 20: y = mlp_act<4>(x); break;
            default: y = mlp_act<5>(x); break;
        }
        out[i] = y;
    }
}

// the f64 truth of the f32 functions (libdevice exp / expm1 / tanh in double: <= 2 ulp of f64, far below an f32 ulp)
__global__ void k_f32_truth(int fn, const uint32_t* in, uint32_t mul, uint32_t add, uint64_t base, double* out, int64_t n) {
    FOR_EACH(i, n) {
        const double x = (double)gen_f32(in, mul, add, base, i);
        out[i] = fn == 0 ? exp(x) : (fn == 1 ? expm1(x) : tanh(x));
    }
}

template <int ACT>
__global__ void k_act2(uint32_t mx, uint32_t ax, uint32_t my, uint32_t ay, uint64_t base, float* ox, float* oy, int64_t n) {
    FOR_EACH(i, n) {
        const float2 r = mlp_act2<ACT>(make_float2(gen_f32(nullptr, mx, ax, base, i), gen_f32(nullptr, my, ay, base, i)));
        ox[i] = r.x;
        oy[i] = r.y;
    }
}

// fn: 0 sin_, 1 cos_, 2 sincos_ (out, out2), 3 log_; 4: log_ of the Box-Muller grid u = (c + 0.5) 2^-32, c = base + i;
// 5: sincos_ of the grid angle 2 pi u (azo_noise / tree_continuous.cuh)
__global__ void k_f64(int fn, const double* in, uint64_t base, double* out, double* out2, int64_t n) {
    FOR_EACH(i, n) {
        double x = fn >= 4 ? ((double)(uint32_t)(base + (uint64_t)i) + 0.5) * 2.3283064365386963e-10 : in[i];
        if (fn == 5) x = 6.283185307179586 * x;
        double s, c;
        switch (fn) {
            case 0: out[i] = det::sin_(x); break;
            case 1: out[i] = det::cos_(x); break;
            case 3: case 4: out[i] = det::log_(x); break;
            default: det::sincos_(x, s, c); out[i] = s; out2[i] = c; break;
        }
    }
}

// which: 0 div_small(a, b), 1 div_tab(a, b), 2 __ddiv_rn(a, b), 3 div_tab_ok(a) as 1.0 / 0.0, 4 sqrt_small(b)
__global__ void k_div(int which, const double* a, const int32_t* b, const double* rcp, const double* sq, int tabn, double* out, int64_t n) {
    FOR_EACH(i, n) {
        double r;
        switch (which) {
            case 0: r = div_small(a[i], b[i], rcp, tabn); break;
            case 1: r = div_tab(a[i], b[i], rcp); break;
            case 2: r = __ddiv_rn(a[i], (double)b[i]); break;
            case 3: r = div_tab_ok(a[i]) ? 1.0 : 0.0; break;
            default: r = sqrt_small(b[i], sq, tabn); break;
        }
        out[i] = r;
    }
}

// ds_decide with W = (W0, W1), cnt = (n0, n1, nn), f = (prior0, prior1, V) per case
__global__ void k_ds_decide(const double* W, const int32_t* cnt, const float* f, const double* rcp, const double* sq, int tabn, double c_uct,
                            int puct_f32, uint32_t* out, int64_t n) {
    DsCtx cx;
    memset(&cx, 0, sizeof cx);
    cx.rcp = rcp; cx.sq = sq; cx.tabn = tabn; cx.c_uct = c_uct; cx.puct_f32 = puct_f32;
    FOR_EACH(i, n) out[i] = ds_decide(cx, W[2 * i], W[2 * i + 1], cnt[3 * i], cnt[3 * i + 1], f[3 * i], f[3 * i + 1], f[3 * i + 2], cnt[3 * i + 2]);
}

// which: 0 rng_block (4 words), 1 rng_select_u32x4 (the four draws idx, idx + stride, ... of stream 0 block 0), 2 philox_draw_x (.x of
// stream 0 block 0, 32-bit draw index)
__global__ void k_philox(int which, uint64_t seed, const int64_t* tree, const int32_t* stream, const int64_t* idx, const int32_t* block,
                         int stride, uint32_t* out, int64_t n) {
    FOR_EACH(i, n) {
        if (which == 0) {
            const u32x4 c = rng_block(seed, tree[i], stream[i], idx[i], block[i]);
            out[4 * i] = c.x; out[4 * i + 1] = c.y; out[4 * i + 2] = c.z; out[4 * i + 3] = c.w;
        } else if (which == 1) {
            rng_select_u32x4(seed, tree[i], (int)idx[i], stride, out + 4 * i);
        } else {
            out[i] = philox_draw_x((uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)tree[i], (uint32_t)((uint64_t)tree[i] >> 32), (uint32_t)idx[i]);
        }
    }
}

__global__ void k_u32_map(const uint32_t* x, const int32_t* m, float* unit, int32_t* index, int64_t n) {
    FOR_EACH(i, n) {
        unit[i] = u32_to_unit(x[i]);
        index[i] = u32_to_index(x[i], m[i]);
    }
}

// one generator per thread, seed[t]; op[k] < 0: random(), 0: a raw output, n > 0: _randbelow(n) (kind 0, CPython); kind 1: torch's
// generator, one double uniform per op.  out[t][k] holds the result of op k as a double.
__global__ void k_mt(int kind, const uint64_t* seed, int ntr, const int32_t* op, int nops, double* out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ntr) return;
    uint32_t mt[TMT_WORDS];
    if (kind == 0) mt_seed_dev(mt, seed[t]); else tmt_seed_dev(mt, seed[t]);
    int mti = (int)mt[MT_N], draws = 0;
    for (int k = 0; k < nops; ++k) {
        double r;
        if (kind == 1) r = tmt_uniform_dev(mt, mti);
        else if (op[k] < 0) r = mt_random_dev(mt, mti, draws);
        else if (op[k] == 0) r = (double)mt_next_dev(mt, mti, draws);
        else r = (double)mt_below_dev(mt, mti, draws, op[k]);
        out[(size_t)t * nops + k] = r;
    }
}

extern "C" {

int probe_f32(int fn, const uint32_t* in, uint32_t mul, uint32_t add, uint64_t base, float* out, int64_t n, cudaStream_t s) {
    k_f32<<<GRID(n), 0, s>>>(fn, in, mul, add, base, out, n);
    return (int)cudaGetLastError();
}
int probe_f32_truth(int fn, const uint32_t* in, uint32_t mul, uint32_t add, uint64_t base, double* out, int64_t n, cudaStream_t s) {
    k_f32_truth<<<GRID(n), 0, s>>>(fn, in, mul, add, base, out, n);
    return (int)cudaGetLastError();
}
int probe_act2(int act, uint32_t mx, uint32_t ax, uint32_t my, uint32_t ay, uint64_t base, float* ox, float* oy, int64_t n, cudaStream_t s) {
    switch (act) {
        case 0: k_act2<0><<<GRID(n), 0, s>>>(mx, ax, my, ay, base, ox, oy, n); break;
        case 1: k_act2<1><<<GRID(n), 0, s>>>(mx, ax, my, ay, base, ox, oy, n); break;
        case 2: k_act2<2><<<GRID(n), 0, s>>>(mx, ax, my, ay, base, ox, oy, n); break;
        case 3: k_act2<3><<<GRID(n), 0, s>>>(mx, ax, my, ay, base, ox, oy, n); break;
        case 4: k_act2<4><<<GRID(n), 0, s>>>(mx, ax, my, ay, base, ox, oy, n); break;
        default: k_act2<5><<<GRID(n), 0, s>>>(mx, ax, my, ay, base, ox, oy, n); break;
    }
    return (int)cudaGetLastError();
}
int probe_f64(int fn, const double* in, uint64_t base, double* out, double* out2, int64_t n, cudaStream_t s) {
    k_f64<<<GRID(n), 0, s>>>(fn, in, base, out, out2, n);
    return (int)cudaGetLastError();
}
int probe_div(int which, const double* a, const int32_t* b, const double* rcp, const double* sq, int tabn, double* out, int64_t n, cudaStream_t s) {
    k_div<<<GRID(n), 0, s>>>(which, a, b, rcp, sq, tabn, out, n);
    return (int)cudaGetLastError();
}
int probe_ds_decide(const double* W, const int32_t* cnt, const float* f, const double* rcp, const double* sq, int tabn, double c_uct,
                    int puct_f32, uint32_t* out, int64_t n, cudaStream_t s) {
    k_ds_decide<<<GRID(n), 0, s>>>(W, cnt, f, rcp, sq, tabn, c_uct, puct_f32, out, n);
    return (int)cudaGetLastError();
}
int probe_philox(int which, uint64_t seed, const int64_t* tree, const int32_t* stream, const int64_t* idx, const int32_t* block, int stride,
                 uint32_t* out, int64_t n, cudaStream_t s) {
    k_philox<<<GRID(n), 0, s>>>(which, seed, tree, stream, idx, block, stride, out, n);
    return (int)cudaGetLastError();
}
int probe_u32_map(const uint32_t* x, const int32_t* m, float* unit, int32_t* index, int64_t n, cudaStream_t s) {
    k_u32_map<<<GRID(n), 0, s>>>(x, m, unit, index, n);
    return (int)cudaGetLastError();
}
int probe_mt(int kind, const uint64_t* seed, int ntr, const int32_t* op, int nops, double* out, cudaStream_t s) {
    k_mt<<<(ntr + 31) / 32, 32, 0, s>>>(kind, seed, ntr, op, nops, out);
    return (int)cudaGetLastError();
}

}  // extern "C"

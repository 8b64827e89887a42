/*
 * azg_oracle.c -- CPU restatement of the alphazero-gym search hot path (see azg_oracle.h).
 * TEST INFRASTRUCTURE ONLY: never linked into, included by, or called from the product path.
 *
 * Build: oracle/Makefile (gcc -O2 -mavx2 -mfma -ffp-contract=off -pthread).  -ffp-contract=off is
 * required: every rounding below is meant literally, fused multiply-adds only where fmaf() is written.
 */
#include "azg_oracle.h"

#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>

#define PENDULUM_R_SCALE 16.2736044 /* mcts.py:20 */

/* ------------------------------------------------------------------------------------------------
 * Philox4x32-10 counter-based generator (Salmon et al., SC'11).  Replaces CPython `random`
 * (helpers.py:51, mcts.py:190-192) and torch's global generator (policies.py:666) by injection:
 * gen_golden.py installs a shim backed by azo_rng_u32/azo_noise into the unmodified reference.
 * counter = (idx_lo, idx_hi ^ (block<<16), tree_lo, tree_hi ^ (stream<<24)), key = seed.
 * ---------------------------------------------------------------------------------------------- */
static inline void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c[0];
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c[2];
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}

static inline void rng_block(uint64_t seed, int64_t tree, int32_t stream, int64_t idx, int32_t block, uint32_t out[4]) {
    out[0] = (uint32_t)idx;
    out[1] = (uint32_t)((uint64_t)idx >> 32) ^ ((uint32_t)block << 16);
    out[2] = (uint32_t)tree;
    out[3] = (uint32_t)((uint64_t)tree >> 32) ^ ((uint32_t)stream << 24);
    philox4x32_10(out, (uint32_t)seed, (uint32_t)(seed >> 32));
}

uint32_t azo_rng_u32(uint64_t seed, int64_t tree, int32_t stream, int64_t idx, int32_t block, int32_t word) {
    uint32_t c[4];
    rng_block(seed, tree, stream, idx, block, c);
    return c[word & 3];
}

/* stream 0: selection draws.  random() -> 24-bit uniform; choice/randint -> multiply-high. */
static inline float u32_to_unit(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-08f; /* 2^-24 */ }
static inline int32_t u32_to_index(uint32_t x, int32_t n) { return (int32_t)(((uint64_t)x * (uint64_t)(uint32_t)n) >> 32); }

/* ------------------------------------------------------------------------------------------------
 * Deterministic math: fixed sequences of IEEE-754 operations (no libm), implemented independently
 * but op-for-op identically in the CUDA engine (csrc/detmath.cuh) so that engine == oracle bit for
 * bit.  Algorithms: Cephes expf/tanhf polynomials; fdlibm __kernel_sin/__kernel_cos/log.
 * ---------------------------------------------------------------------------------------------- */
static inline float f32_from_bits(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
static inline uint32_t f32_bits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }

/* exp(r)-1 for |r| <= 0.5*ln2 (+rounding slack): r + r^2 * P(r) */
static inline float expm1_poly(float r) {
    float p = 1.9875691500E-4f;
    p = fmaf(p, r, 1.3981999507E-3f);
    p = fmaf(p, r, 8.3334519073E-3f);
    p = fmaf(p, r, 4.1665795894E-2f);
    p = fmaf(p, r, 1.6666665459E-1f);
    p = fmaf(p, r, 5.0000001201E-1f);
    float z = r * r;
    return fmaf(p, z, r);
}

static inline float exp_reduce(float x, float* n_out) {
    float n = rintf(x * 1.44269504088896341f);
    float r = fmaf(n, -0.693359375f, x);
    r = fmaf(n, 2.12194440e-4f, r);
    *n_out = n;
    return r;
}

float azo_det_expf(float x) {
    if (!(x <= 88.0f)) return (x != x) ? x : INFINITY;
    if (x < -87.0f) return 0.0f; /* flushes the denormal tail; documented */
    float n;
    float r = exp_reduce(x, &n);
    float y = expm1_poly(r) + 1.0f;
    return f32_from_bits(f32_bits(y) + ((uint32_t)(int32_t)n << 23));
}

float azo_det_expm1f(float x) {
    if (x != x) return x;
    if (x < -17.5f) return -1.0f;
    if (x > 88.0f) return INFINITY;
    float n;
    float r = exp_reduce(x, &n);
    float p = expm1_poly(r);
    if (n == 0.0f) return p;
    float t = f32_from_bits((uint32_t)((int32_t)n + 127) << 23); /* 2^n, n in [-25, 127] */
    return fmaf(p, t, t - 1.0f);
}

float azo_det_tanhf(float x) {
    float ax = fabsf(x);
    float y;
    if (ax != ax) return x;
    if (ax >= 9.1f) {
        y = 1.0f;
    } else if (ax >= 0.625f) {
        float e = azo_det_expf(ax + ax);
        y = 1.0f - 2.0f / (e + 1.0f);
    } else {
        float z = ax * ax;
        float p = -5.70498872745E-3f;
        p = fmaf(p, z, 2.06390887954E-2f);
        p = fmaf(p, z, -5.37397155531E-2f);
        p = fmaf(p, z, 1.33314422036E-1f);
        p = fmaf(p, z, -3.33332819422E-1f);
        y = fmaf(p * z, ax, ax);
    }
    return copysignf(y, x);
}

static inline double ksin(double x, double y) {
    const double S1 = -1.66666666666666324348e-01, S2 = 8.33333333332248946124e-03, S3 = -1.98412698298579493134e-04,
                 S4 = 2.75573137070700676789e-06, S5 = -2.50507602534068634195e-08, S6 = 1.58969099521155010221e-10;
    double z = x * x;
    double w = z * z;
    double r = (S2 + z * (S3 + z * S4)) + (z * w) * (S5 + z * S6);
    double v = z * x;
    return x - ((z * (0.5 * y - v * r) - y) - v * S1);
}

static inline double kcos(double x, double y) {
    const double C1 = 4.16666666666666019037e-02, C2 = -1.38888888888741095749e-03, C3 = 2.48015872894767294178e-05,
                 C4 = -2.75573143513906633035e-07, C5 = 2.08757232129817482790e-09, C6 = -1.13596475577881948265e-11;
    double z = x * x;
    double w = z * z;
    double r = z * (C1 + z * (C2 + z * C3)) + (w * w) * (C4 + z * (C5 + z * C6));
    double hz = 0.5 * z;
    double w1 = 1.0 - hz;
    return w1 + (((1.0 - w1) - hz) + (z * r - x * y));
}

/* Cody-Waite reduction with 2x33-bit pieces of pi/2 (valid for |x| < 2^20 * pi/2) */
static inline int rem_pio2(double x, double* y0, double* y1) {
    const double invpio2 = 6.36619772367581382433e-01, pio2_1 = 1.57079632673412561417e+00,
                 pio2_2 = 6.07710050630396597660e-11, pio2_2t = 2.02226624879595063154e-21;
    double fn = rint(x * invpio2);
    double t = x - fn * pio2_1;
    double w = fn * pio2_2;
    double r = t - w;
    w = fn * pio2_2t - ((t - r) - w);
    *y0 = r - w;
    *y1 = (r - *y0) - w;
    return (int)fn;
}

double azo_det_sin(double x) {
    double y0, y1;
    int n = rem_pio2(x, &y0, &y1);
    switch (n & 3) {
        case 0: return ksin(y0, y1);
        case 1: return kcos(y0, y1);
        case 2: return -ksin(y0, y1);
        default: return -kcos(y0, y1);
    }
}

double azo_det_cos(double x) {
    double y0, y1;
    int n = rem_pio2(x, &y0, &y1);
    switch (n & 3) {
        case 0: return kcos(y0, y1);
        case 1: return -ksin(y0, y1);
        case 2: return -kcos(y0, y1);
        default: return ksin(y0, y1);
    }
}

/* log(x) for normal positive x (fdlibm e_log.c evaluation scheme) */
double azo_det_log(double x) {
    const double ln2_hi = 6.93147180369123816490e-01, ln2_lo = 1.90821492927058770002e-10,
                 Lg1 = 6.666666666666735130e-01, Lg2 = 3.999999999940941908e-01, Lg3 = 2.857142874366239149e-01,
                 Lg4 = 2.222219843214978396e-01, Lg5 = 1.818357216161805012e-01, Lg6 = 1.531383769920937332e-01,
                 Lg7 = 1.479819860511658591e-01;
    uint64_t bits;
    memcpy(&bits, &x, 8);
    uint32_t hx = (uint32_t)(bits >> 32);
    hx += 0x3ff00000u - 0x3fe6a09eu;
    int32_t k = (int32_t)(hx >> 20) - 0x3ff;
    hx = (hx & 0x000fffffu) + 0x3fe6a09eu;
    bits = ((uint64_t)hx << 32) | (bits & 0xffffffffull);
    memcpy(&x, &bits, 8);
    double f = x - 1.0;
    double hfsq = 0.5 * f * f;
    double s = f / (2.0 + f);
    double z = s * s;
    double w = z * z;
    double t1 = w * (Lg2 + w * (Lg4 + w * Lg6));
    double t2 = z * (Lg1 + w * (Lg3 + w * (Lg5 + w * Lg7)));
    double R = t2 + t1;
    double dk = (double)k;
    return ((((s * (hfsq + R)) + dk * ln2_lo) - hfsq) + f) + dk * ln2_hi;
}

/* stream 1: noise for progressive-widening insert j.  block 0 word 0 -> component uniform;
 * block 1+b words 0,1 -> Box-Muller pair (z[2b], z[2b+1]).  Always deterministic math. */
void azo_noise(uint64_t seed, int64_t tree, int64_t j, int32_t K, float* u_comp, float* z) {
    uint32_t c[4];
    rng_block(seed, tree, 1, j, 0, c);
    *u_comp = u32_to_unit(c[0]);
    for (int b = 0; 2 * b < K; ++b) {
        rng_block(seed, tree, 1, j, 1 + b, c);
        double u1 = ((double)c[0] + 0.5) * 2.3283064365386963e-10; /* 2^-32 */
        double u2 = ((double)c[1] + 0.5) * 2.3283064365386963e-10;
        double rad = sqrt(-2.0 * azo_det_log(u1));
        double ang = 6.283185307179586 * u2;
        z[2 * b] = (float)(rad * azo_det_cos(ang));
        if (2 * b + 1 < K) z[2 * b + 1] = (float)(rad * azo_det_sin(ang));
    }
}

/* ------------------------------------------------------------------------------------------------
 * Network (policies.py): trunk Linear+act x n_hidden, value_head Linear(H,1), dist_head Linear(H,P).
 * Summation order is part of the contract: acc = bias; acc = fmaf(w[j][k], x[k], acc) for k ascending.
 * ---------------------------------------------------------------------------------------------- */
int32_t azo_head_dim(const azo_config* c) {
    if (c->variant == AZO_DISCRETE) return c->num_actions;
    return c->num_components > 1 ? 3 * c->num_components : 2; /* policies.py:587-588 / :434 (action_dim = 1) */
}

int64_t azo_num_weights(const azo_config* c) {
    int64_t H = c->hidden, n = (int64_t)c->state_dim * H + H;
    for (int l = 1; l < c->n_hidden; ++l) n += H * H + H;
    n += H + 1;
    n += (int64_t)azo_head_dim(c) * H + azo_head_dim(c);
    return n;
}

typedef struct {
    int S, H, L, P;
    float* wt[AZO_MAX_LAYERS]; /* transposed trunk weights [K][H] (k-major so the j loop vectorises) */
    const float* b[AZO_MAX_LAYERS];
    const float *wv, *bv, *wd, *bd;
    float* owned;
    /* AZO_EVAL_Q8: digit planes [3][H][H] (row j, column k) and per-output scale of every hidden layer l >= 1 */
    int8_t* qd[AZO_MAX_LAYERS];
    float* qcw[AZO_MAX_LAYERS];
} net_t;

static inline int biased_exp_clamped(float f) {
    int e = (int)((f32_bits(f) >> 23) & 0xFF);
    return e < 32 ? 32 : (e > 200 ? 200 : e);
}
/* cvt.rni.s32.f32: round to nearest even, saturating, NaN -> 0 */
static inline int32_t rni_sat(float t) {
    if (t != t) return 0;
    if (t >= 2147483648.0f) return INT32_MAX;
    if (t <= -2147483648.0f) return INT32_MIN;
    return (int32_t)rintf(t);
}

/* balanced signed base-256 digits of q (|q| <= 8355711): bytes of (q + 0x8080) with the two low bytes' top bit flipped */
static inline void q8_digits(int32_t q, int8_t* hi, int8_t* mid, int8_t* lo) {
    const uint32_t t = ((uint32_t)q + 0x8080u) ^ 0x8080u;
    *lo = (int8_t)(t & 0xFF);
    *mid = (int8_t)((t >> 8) & 0xFF);
    *hi = (int8_t)((t >> 16) & 0xFF);
}
/* biased exponent e such that |v| * 2^(149-e) <= 8355711 for every |v| <= vmax (1.004 keeps the top digit in int8) */
static inline int q8_exponent(float vmax) { return biased_exp_clamped(vmax * 1.004f); }

static void net_quantize(net_t* n, const float* w_state_dict) {
    const int H = n->H;
    const float* w = w_state_dict + (size_t)n->S * H + H;
    for (int l = 1; l < n->L; ++l) {
        n->qd[l] = (int8_t*)malloc((size_t)3 * H * H);
        n->qcw[l] = (float*)malloc((size_t)H * sizeof(float));
        for (int j = 0; j < H; ++j) {
            float wmax = 0.0f;
            for (int k = 0; k < H; ++k) wmax = fmaxf(wmax, fabsf(w[(size_t)j * H + k]));
            const int e = q8_exponent(wmax);
            const float sc = f32_from_bits((uint32_t)(276 - e) << 23); /* 2^(149-e) */
            n->qcw[l][j] = f32_from_bits((uint32_t)(e - 6) << 23);      /* 2^(e-133) = 2^16 / sc */
            for (int k = 0; k < H; ++k)
                q8_digits(rni_sat(w[(size_t)j * H + k] * sc), &n->qd[l][(size_t)j * H + k], &n->qd[l][(size_t)H * H + (size_t)j * H + k],
                          &n->qd[l][(size_t)2 * H * H + (size_t)j * H + k]);
        }
        w += (size_t)H * H + H;
    }
}

static int net_init(net_t* n, const azo_config* c, const float* w, int64_t nw) {
    if (c->n_hidden < 1 || c->n_hidden > AZO_MAX_LAYERS || c->hidden < 1 || nw != azo_num_weights(c)) return -2;
    n->S = c->state_dim; n->H = c->hidden; n->L = c->n_hidden; n->P = azo_head_dim(c);
    const float* w0 = w;
    size_t tot = (size_t)n->S * n->H + (size_t)(n->L - 1) * n->H * n->H;
    n->owned = (float*)malloc(tot * sizeof(float));
    float* dst = n->owned;
    for (int l = 0; l < n->L; ++l) {
        int K = l == 0 ? n->S : n->H;
        n->wt[l] = dst;
        for (int j = 0; j < n->H; ++j)
            for (int k = 0; k < K; ++k) dst[(size_t)k * n->H + j] = w[(size_t)j * K + k];
        dst += (size_t)K * n->H;
        w += (size_t)K * n->H;
        n->b[l] = w;
        w += n->H;
    }
    n->wv = w; w += n->H;
    n->bv = w; w += 1;
    n->wd = w; w += (size_t)n->P * n->H;
    n->bd = w;
    for (int l = 0; l < AZO_MAX_LAYERS; ++l) { n->qd[l] = NULL; n->qcw[l] = NULL; }
    if (c->eval_mode == AZO_EVAL_Q8) {
        if (n->H % 32 != 0) return -2;
        net_quantize(n, w0);
    }
    return 0;
}

static void net_free(net_t* n) {
    free(n->owned); n->owned = NULL;
    for (int l = 0; l < AZO_MAX_LAYERS; ++l) { free(n->qd[l]); free(n->qcw[l]); n->qd[l] = NULL; n->qcw[l] = NULL; }
}

static inline float act_fn(const azo_config* c, float v) {
    if (c->activation == AZO_ACT_RELU) return v > 0.0f ? v : 0.0f;
    if (c->activation == AZO_ACT_LEAKYRELU) return v > 0.0f ? v : v * 0.01f;
    if (c->activation == AZO_ACT_RELU6) {
        /* a NaN is a missing operand of fmaxf, as on the GPU: 0.  (glibc's fmaxf returns NaN for a signaling NaN, and fminf
         * then returns 6; tests/test_primitives_gpu.py compares every f32 input.) */
        if (v != v) return 0.0f;
        return fminf(fmaxf(v, 0.0f), 6.0f);
    }
    if (c->activation == AZO_ACT_SILU) {
        if (v != v) return v;
        const float e = c->math_mode == AZO_MATH_DET ? azo_det_expf(-v) : expf(-v);
        volatile float d = 1.0f + e;
        return v / d;
    }
    if (c->activation == AZO_ACT_HARDSWISH) {
        volatile float t = v + 3.0f;
        volatile float m = v * fminf(fmaxf(t, 0.0f), 6.0f);
        return m / 6.0f;
    }
    /* ELU alpha=1 (ContinuousPolicy.yaml:9): x > 0 ? x : expm1(x) */
    if (v > 0.0f) return v;
    return c->math_mode == AZO_MATH_DET ? azo_det_expm1f(v) : expm1f(v);
}

/* one hidden layer of the AZO_EVAL_Q8 contract (azg_oracle.h) */
static void q8_layer(const net_t* n, const azo_config* c, int l, const float* in, float* out) {
    const int H = n->H;
    int8_t xh[1024], xm[1024], xl[1024];
    float m = 0.0f;
    for (int k = 0; k < H; ++k) m = fmaxf(m, fabsf(in[k]));
    const int e = q8_exponent(m);
    const float sx = f32_from_bits((uint32_t)(276 - e) << 23); /* 2^(149-e) */
    const float cx = f32_from_bits((uint32_t)(e - 22) << 23);  /* 2^(e-149) */
    for (int k = 0; k < H; ++k) q8_digits(rni_sat(in[k] * sx), &xh[k], &xm[k], &xl[k]);
    const int8_t* dh = n->qd[l];
    const int8_t* dm = dh + (size_t)H * H;
    const int8_t* dl = dm + (size_t)H * H;
    for (int j = 0; j < H; ++j) {
        const int8_t* wh = dh + (size_t)j * H;
        const int8_t* wm = dm + (size_t)j * H;
        const int8_t* wl = dl + (size_t)j * H;
        int32_t PA = 0, PB = 0, PC = 0;
        for (int k = 0; k < H; ++k) {
            const int32_t a2 = xh[k], a1 = xm[k], a0 = xl[k];
            PA += a2 * wh[k];
            PB += a2 * wm[k] + a1 * wh[k];
            PC += a2 * wl[k] + a1 * wm[k] + a0 * wh[k];
        }
        float u = fmaf((float)PA, 256.0f, (float)PB);
        u = fmaf(u, 256.0f, (float)PC);
        out[j] = act_fn(c, fmaf(u, cx * n->qcw[l][j], n->b[l][j]));
    }
}

static inline float q8_head(const float* w, const float* in, int H, float bias) {
    float part[32];
    const int nq = H / 32;
    for (int q = 0; q < nq; ++q) {
        float s = 0.0f;
        for (int k = 32 * q; k < 32 * q + 32; ++k) s = fmaf(in[k], w[k], s);
        part[q] = s;
    }
    for (int span = 1; span < nq; span *= 2)
        for (int q = 0; q + span < nq; q += 2 * span) part[q] = part[q] + part[q + span];
    return part[0] + bias;
}

static void net_forward(const net_t* n, const azo_config* c, const float* x, float* V, float* head) {
    float h0[1024], h1[1024];
    float* in = h0;
    float* out = h1;
    const int H = n->H;
    const int q8 = c->eval_mode == AZO_EVAL_Q8;
    for (int k = 0; k < n->S; ++k) in[k] = x[k];
    for (int l = 0; l < n->L; ++l) {
        if (q8 && l > 0) {
            q8_layer(n, c, l, in, out);
        } else {
            int K = l == 0 ? n->S : H;
            const float* wt = n->wt[l];
            for (int j = 0; j < H; ++j) out[j] = n->b[l][j];
            for (int k = 0; k < K; ++k) {
                const float xk = in[k];
                const float* wr = wt + (size_t)k * H;
                for (int j = 0; j < H; ++j) out[j] = __builtin_fmaf(wr[j], xk, out[j]);
            }
            for (int j = 0; j < H; ++j) out[j] = act_fn(c, out[j]);
        }
        float* t = in; in = out; out = t;
    }
    if (q8) {
        *V = q8_head(n->wv, in, H, n->bv[0]);
        for (int p = 0; p < n->P; ++p) head[p] = q8_head(n->wd + (size_t)p * H, in, H, n->bd[p]);
        return;
    }
    float acc = n->bv[0];
    for (int k = 0; k < H; ++k) acc = fmaf(n->wv[k], in[k], acc);
    *V = acc;
    for (int p = 0; p < n->P; ++p) {
        acc = n->bd[p];
        const float* wr = n->wd + (size_t)p * H;
        for (int k = 0; k < H; ++k) acc = fmaf(wr[k], in[k], acc);
        head[p] = acc;
    }
}

void azo_mlp_forward(const azo_config* cfg, const float* weights, int32_t n, const float* x, float* out_V, float* out_head) {
    net_t net;
    if (cfg->hidden > 1024 || net_init(&net, cfg, weights, azo_num_weights(cfg))) return;
    for (int i = 0; i < n; ++i) net_forward(&net, cfg, x + (size_t)i * net.S, out_V + i, out_head + (size_t)i * net.P);
    net_free(&net);
}

static inline float m_expf(const azo_config* c, float x) { return c->math_mode == AZO_MATH_DET ? azo_det_expf(x) : expf(x); }

/* softmax in index order (policies.py:352 F.softmax; torch Categorical(logits) probs) */
static void softmax_seq(const azo_config* c, const float* l, int n, float* p) {
    float m = l[0];
    for (int i = 1; i < n; ++i) m = l[i] > m ? l[i] : m;
    float s = 0.0f;
    for (int i = 0; i < n; ++i) { p[i] = m_expf(c, l[i] - m); s += p[i]; }
    for (int i = 0; i < n; ++i) p[i] = p[i] / s;
}

void azo_head_post(const azo_config* c, const float* raw, float* out) {
    if (c->variant == AZO_DISCRETE) { softmax_seq(c, raw, c->num_actions, out); return; }
    const int K = c->num_components;
    /* policies.py:617-631 (GMM) / :451-458 (Normal): mu | clamp(log_std).exp() | mixture logits */
    for (int k = 0; k < K; ++k) {
        out[k] = raw[k];
        float ls = raw[K + k];
        ls = ls < c->log_std_min ? c->log_std_min : ls;
        ls = ls > c->log_std_max ? c->log_std_max : ls;
        out[K + k] = m_expf(c, ls);
    }
    if (K > 1) softmax_seq(c, raw + 2 * K, K, out + 2 * K);
    else out[2] = 1.0f;
}

/* MixtureSameFamily.sample: component by inverse CDF on u (injected in place of torch.multinomial),
 * x = z*sigma + mu (torch.normal: mul then add), action = bound*tanh(x) (distributions.py:50-63). */
float azo_sample_action(const azo_config* c, const float* head, float u, const float* z) {
    const int K = c->num_components;
    int k = 0;
    if (K > 1) {
        float cum = head[2 * K];
        while (k < K - 1 && !(u < cum)) { ++k; cum += head[2 * K + k]; }
    }
    float x = z[k] * head[K + k] + head[k];
    float t = c->math_mode == AZO_MATH_DET ? azo_det_tanhf(x) : tanhf(x);
    return c->action_bound > 0.0f ? c->action_bound * t : x; /* policies.py:660-663: unbounded -> plain Normal */
}

/* ------------------------------------------------------------------------------------------------
 * Environment dynamics (gym classic_control, restated; SURVEY 8c).
 * ---------------------------------------------------------------------------------------------- */
static inline double m_sin(const azo_config* c, double x) { return c->math_mode == AZO_MATH_DET ? azo_det_sin(x) : sin(x); }
static inline double m_cos(const azo_config* c, double x) { return c->math_mode == AZO_MATH_DET ? azo_det_cos(x) : cos(x); }

static int cartpole_step(const azo_config* c, const double* s, int action, double* o, double* reward) {
    const double gravity = 9.8, masscart = 1.0, masspole = 0.1, length = 0.5, force_mag = 10.0, tau = 0.02;
    const double total_mass = masspole + masscart, polemass_length = masspole * length;
    const double theta_thr = 12 * 2 * 3.141592653589793 / 360, x_thr = 2.4;
    double x = s[0], x_dot = s[1], theta = s[2], theta_dot = s[3];
    double force = action == 1 ? force_mag : -force_mag;
    double costheta = m_cos(c, theta), sintheta = m_sin(c, theta);
    double temp = (force + polemass_length * (theta_dot * theta_dot) * sintheta) / total_mass;
    double thetaacc = (gravity * sintheta - costheta * temp) / (length * (4.0 / 3.0 - masspole * (costheta * costheta) / total_mass));
    double xacc = temp - polemass_length * thetaacc * costheta / total_mass;
    x = x + tau * x_dot;
    x_dot = x_dot + tau * xacc;
    theta = theta + tau * theta_dot;
    theta_dot = theta_dot + tau * thetaacc;
    o[0] = x; o[1] = x_dot; o[2] = theta; o[3] = theta_dot;
    *reward = 1.0;
    return x < -x_thr || x > x_thr || theta < -theta_thr || theta > theta_thr;
}

static inline double py_mod(double a, double b) {
    double r = fmod(a, b);
    if (r != 0.0) { if ((b < 0) != (r < 0)) r += b; } else r = copysign(0.0, b);
    return r;
}

static int pendulum_step(const azo_config* c, const double* s, float action, double* o, double* reward) {
    const double max_speed = 8, dt = 0.05, g = 10.0, m = 1.0, l = 1.0, pi = 3.141592653589793;
    double th = s[0], thdot = s[1];
    float uf = action < -2.0f ? -2.0f : (action > 2.0f ? 2.0f : action); /* np.clip on the f32 action */
    double u = (double)uf;                                               /* numpy-1.x promotion (SURVEY 8c) */
    double an = py_mod(th + pi, 2 * pi) - pi;
    double costs = an * an + 0.1 * (thdot * thdot) + 0.001 * (u * u);
    double newthdot = thdot + (-3 * g / (2 * l) * m_sin(c, th + pi) + 3.0 / (m * (l * l)) * u) * dt;
    double newth = th + newthdot * dt;
    newthdot = newthdot < -max_speed ? -max_speed : (newthdot > max_speed ? max_speed : newthdot);
    o[0] = newth; o[1] = newthdot;
    *reward = -costs;
    return 0;
}

static void pendulum_obs(const azo_config* c, const double* s, float* obs) {
    obs[0] = (float)m_cos(c, s[0]);
    obs[1] = (float)m_sin(c, s[0]);
    obs[2] = (float)s[1];
}

/* MountainCarContinuous-v0.  The f32 action enters f64 arithmetic exactly (numpy-1.x promotion); force = min(max(a, -1.0), 1.0) with
 * Python's max / min (a NaN passes, -0 stays -0); velocity + ((force * power) - (0.0025 * cos(3 * position))); the left wall sets
 * velocity to +0; done = position >= 0.45 and velocity >= 0; reward (done ? 100.0 : 0.0) - pow(a, 2) * 0.1 on the unclipped action
 * (0 - x with the int 0 is 0.0 - x: +0 for a zero action; pow(a, 2) of an f32 is exact in f64). */
static int mountain_car_continuous_step(const azo_config* c, const double* s, float action, double* o, double* reward) {
    const double min_position = -1.2, max_position = 0.6, max_speed = 0.07, goal_position = 0.45, power = 0.0015;
    double pos = s[0], vel = s[1];
    const double a = (double)action;
    double force = -1.0 > a ? -1.0 : a;
    force = 1.0 < force ? 1.0 : force;
    vel = vel + (force * power - 0.0025 * m_cos(c, 3 * pos));
    if (vel > max_speed) vel = max_speed;
    if (vel < -max_speed) vel = -max_speed;
    pos = pos + vel;
    if (pos > max_position) pos = max_position;
    if (pos < min_position) pos = min_position;
    if (pos == min_position && vel < 0) vel = 0.0;
    const int done = pos >= goal_position && vel >= 0.0;
    *reward = (done ? 100.0 : 0.0) - (a * a) * 0.1;
    o[0] = pos; o[1] = vel;
    return done;
}

/* MountainCar-v0.  velocity += (action - 1) * force + cos(3 * position) * (-gravity), the right-hand side summed first ((action - 1) *
 * force is an int times a float); np.clip on velocity and position (a NaN passes, -0 stays -0); the left wall stores the int 0 (+0 from
 * then on); done = position >= 0.5 and velocity >= 0 (false for a NaN); reward -1.0 on every step. */
static int mountain_car_step(const azo_config* c, const double* s, int action, double* o, double* reward) {
    const double min_position = -1.2, max_position = 0.6, max_speed = 0.07, goal_position = 0.5, force = 0.001, gravity = 0.0025;
    double pos = s[0], vel = s[1];
    vel = vel + ((double)(action - 1) * force + m_cos(c, 3 * pos) * -gravity);
    vel = vel < -max_speed ? -max_speed : (vel > max_speed ? max_speed : vel);
    pos = pos + vel;
    pos = pos < min_position ? min_position : (pos > max_position ? max_position : pos);
    if (pos == min_position && vel < 0) vel = 0.0;
    *reward = -1.0;
    o[0] = pos; o[1] = vel;
    return pos >= goal_position && vel >= 0.0;
}

/* Acrobot-v1 (book dynamics, no torque noise) */
#define ACROBOT_WRAP_CAP 64 /* iterations per wrap loop, as in the engine (env.cuh) */

static void acrobot_dsdt(const azo_config* c, const double* s, double a, double* d) {
    const double m1 = 1.0, m2 = 1.0, l1 = 1.0, lc1 = 0.5, lc2 = 0.5, I1 = 1.0, I2 = 1.0, g = 9.8, pi = 3.141592653589793;
    const double theta1 = s[0], theta2 = s[1], dtheta1 = s[2], dtheta2 = s[3];
    const double c2 = m_cos(c, theta2), s2 = m_sin(c, theta2);
    const double d1 = m1 * (lc1 * lc1) + m2 * (l1 * l1 + lc2 * lc2 + 2 * l1 * lc2 * c2) + I1 + I2;
    const double d2 = m2 * (lc2 * lc2 + l1 * lc2 * c2) + I2;
    const double phi2 = m2 * lc2 * g * m_cos(c, theta1 + theta2 - pi / 2.);
    const double phi1 = -m2 * l1 * lc2 * (dtheta2 * dtheta2) * s2 - 2 * m2 * l1 * lc2 * dtheta2 * dtheta1 * s2 +
                        (m1 * lc1 + m2 * l1) * g * m_cos(c, theta1 - pi / 2) + phi2;
    const double ddtheta2 = (a + d2 / d1 * phi1 - m2 * l1 * lc2 * (dtheta1 * dtheta1) * s2 - phi2) / (m2 * (lc2 * lc2) + I2 - (d2 * d2) / d1);
    const double ddtheta1 = -(d2 * ddtheta2 + phi1) / d1;
    d[0] = dtheta1; d[1] = dtheta2; d[2] = ddtheta1; d[3] = ddtheta2;
}

/* gym's wrap with each loop capped at ACROBOT_WRAP_CAP iterations (*capped = 1 when a loop would go on) */
static double acrobot_wrap(double x, int* capped) {
    const double pi = 3.141592653589793, diff = pi - -pi;
    for (int k = 0; x > pi; ++k) {
        if (k == ACROBOT_WRAP_CAP) { *capped = 1; return x; }
        x = x - diff;
    }
    for (int k = 0; x < -pi; ++k) {
        if (k == ACROBOT_WRAP_CAP) { *capped = 1; return x; }
        x = x + diff;
    }
    return x;
}

/* min(max(x, m), M) with Python's builtins: a NaN passes, -0 stays -0 */
static double acrobot_bound(double x, double m, double M) {
    x = m > x ? m : x;
    return M < x ? M : x;
}

/* one step: RK4 over [0, dt] of the book dynamics, wrap, bound; returns terminal, or AZO_ERR_WRAP when a wrap loop reached its cap */
static int acrobot_step(const azo_config* c, const double* s, int action, double* o, double* reward) {
    const double dt = .2, pi = 3.141592653589793, MAX_VEL_1 = 4 * pi, MAX_VEL_2 = 9 * pi;
    const double torque = action == 0 ? -1.0 : (action == 1 ? 0.0 : 1.0);
    const double dt2 = dt / 2.0;
    double k1[4], k2[4], k3[4], k4[4], y[4];
    int capped = 0;
    acrobot_dsdt(c, s, torque, k1);
    for (int i = 0; i < 4; ++i) y[i] = s[i] + dt2 * k1[i];
    acrobot_dsdt(c, y, torque, k2);
    for (int i = 0; i < 4; ++i) y[i] = s[i] + dt2 * k2[i];
    acrobot_dsdt(c, y, torque, k3);
    for (int i = 0; i < 4; ++i) y[i] = s[i] + dt * k3[i];
    acrobot_dsdt(c, y, torque, k4);
    for (int i = 0; i < 4; ++i) o[i] = s[i] + dt / 6.0 * (k1[i] + 2 * k2[i] + 2 * k3[i] + k4[i]);
    o[0] = acrobot_wrap(o[0], &capped);
    o[1] = acrobot_wrap(o[1], &capped);
    o[2] = acrobot_bound(o[2], -MAX_VEL_1, MAX_VEL_1);
    o[3] = acrobot_bound(o[3], -MAX_VEL_2, MAX_VEL_2);
    const int terminal = -m_cos(c, o[0]) - m_cos(c, o[1] + o[0]) > 1.;
    *reward = terminal ? 0.0 : -1.0;
    return capped ? AZO_ERR_WRAP : terminal;
}

/* _get_ob of a hidden state, each entry rounded to f32 */
static void acrobot_obs(const azo_config* c, const double* s, float* x) {
    x[0] = (float)m_cos(c, s[0]); x[1] = (float)m_sin(c, s[0]); x[2] = (float)m_cos(c, s[1]); x[3] = (float)m_sin(c, s[1]);
    x[4] = (float)s[2]; x[5] = (float)s[3];
}

/* The env dispatch: the only code that depends on which env a config steps.  A discrete action arrives as its index in a float. */
#define ENV_MAX_OBS 6 /* widest observation (Acrobot) */

static int env_hidden_dim(const azo_config* c) {
    switch (c->env) {
        case AZO_ENV_MOUNTAIN_CAR_CONTINUOUS: case AZO_ENV_MOUNTAIN_CAR: return 2;
        case AZO_ENV_ACROBOT: return 4;
        default: return c->variant == AZO_DISCRETE ? 4 : 2;
    }
}

static int env_step(const azo_config* c, const double* s, float action, double* o, double* reward) {
    switch (c->env) {
        case AZO_ENV_MOUNTAIN_CAR_CONTINUOUS: return mountain_car_continuous_step(c, s, action, o, reward);
        case AZO_ENV_MOUNTAIN_CAR: return mountain_car_step(c, s, (int)action, o, reward);
        case AZO_ENV_ACROBOT: return acrobot_step(c, s, (int)action, o, reward);
        default: return c->variant == AZO_DISCRETE ? cartpole_step(c, s, (int)action, o, reward) : pendulum_step(c, s, action, o, reward);
    }
}

/* the network input of a hidden state: Pendulum (cos th, sin th, thdot), Acrobot _get_ob, the others the state itself (f32) */
static void env_obs(const azo_config* c, const double* s, float* x) {
    if (c->env == AZO_ENV_ACROBOT) acrobot_obs(c, s, x);
    else if (c->env == AZO_ENV_DEFAULT && c->variant == AZO_CONTINUOUS) pendulum_obs(c, s, x);
    else for (int i = 0; i < env_hidden_dim(c); ++i) x[i] = (float)s[i];
}

int azo_env_step(const azo_config* c, const double* s_in, float action, double* s_out, double* reward, float* obs) {
    const int term = env_step(c, s_in, action, s_out, reward);
    if (obs) env_obs(c, s_out, obs);
    return term;
}

void azo_obs(const azo_config* c, const double* s, float* obs) { env_obs(c, s, obs); }

int32_t azo_pw_limit(double c_pw, double kappa, int32_t n) { return (int32_t)ceil(c_pw * pow((double)(n + 1), kappa)); }

/* ------------------------------------------------------------------------------------------------
 * Selection helpers.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    uint64_t seed; int64_t tree; int64_t draws; int64_t pw; int mt_mode; int mti; uint32_t mt[624];
    /* AZO_RNG_MT19937, continuous search: torch's CPU generator (see torch_sample_action) */
    int tmti; uint32_t tmt[624]; int tcache_valid; double tcache; int64_t tdraws;
} rng_t;

static inline uint32_t rng_next(rng_t* g) { return azo_rng_u32(g->seed, g->tree, 0, g->draws++, 0, 0); }

/* AZO_RNG_MT19937 (config.rng_mode = 1; SURVEY 8f rank 4): the selection draws come from CPython's own generator, so that an
 * UN-SHIMMED reference run -- stock `random` module, `random.seed(seed + tree)` right before MCTSDiscrete.search -- is reproduced:
 * MT19937 seeded by init_by_array (CPython random_seed with an int), random() = 53 bits from two outputs, choice / randint =
 * _randbelow_with_getrandbits (k = n.bit_length(); draw the top k bits until < n).  `draws` counts generator outputs. */
static void mt_init_genrand(uint32_t* mt, uint32_t s) {
    mt[0] = s;
    for (int i = 1; i < 624; ++i) mt[i] = 1812433253u * (mt[i - 1] ^ (mt[i - 1] >> 30)) + (uint32_t)i;
}
static void mt_seed(rng_t* g, uint64_t seed) {
    uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    const int klen = key[1] ? 2 : 1;
    uint32_t* mt = g->mt;
    mt_init_genrand(mt, 19650218u);
    int i = 1, j = 0;
    for (int k = 624 > klen ? 624 : klen; k; --k) {
        mt[i] = (mt[i] ^ ((mt[i - 1] ^ (mt[i - 1] >> 30)) * 1664525u)) + key[j] + (uint32_t)j;
        ++i; ++j;
        if (i >= 624) { mt[0] = mt[623]; i = 1; }
        if (j >= klen) j = 0;
    }
    for (int k = 623; k; --k) {
        mt[i] = (mt[i] ^ ((mt[i - 1] ^ (mt[i - 1] >> 30)) * 1566083941u)) - (uint32_t)i;
        ++i;
        if (i >= 624) { mt[0] = mt[623]; i = 1; }
    }
    mt[0] = 0x80000000u;
    g->mti = 624;
}
static uint32_t mt_next(rng_t* g) {
    uint32_t* mt = g->mt;
    if (g->mti >= 624) {
        int kk;
        uint32_t y;
        for (kk = 0; kk < 624 - 397; ++kk) { y = (mt[kk] & 0x80000000u) | (mt[kk + 1] & 0x7fffffffu); mt[kk] = mt[kk + 397] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u); }
        for (; kk < 623; ++kk) { y = (mt[kk] & 0x80000000u) | (mt[kk + 1] & 0x7fffffffu); mt[kk] = mt[kk + (397 - 624)] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u); }
        y = (mt[623] & 0x80000000u) | (mt[0] & 0x7fffffffu);
        mt[623] = mt[396] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
        g->mti = 0;
    }
    uint32_t y = mt[g->mti++];
    y ^= y >> 11; y ^= (y << 7) & 0x9d2c5680u; y ^= (y << 15) & 0xefc60000u; y ^= y >> 18;
    g->draws++;
    return y;
}
/* ---- AZO_RNG_MT19937, continuous search: the action noise comes from torch's global CPU generator exactly as an UN-WRAPPED
 * `model.sample_action` consumes it after `torch.manual_seed(seed + tree)` (policies.py:656-669 / :488-499; measured against
 * torch 2.11 in the build container, oracle/gen_golden.py "pendulum_mt_*"):
 *   generator   at::mt19937 seeded with init_genrand((uint32) seed); random64() = (out1 << 32) | out2
 *   uniform     (random64() & (2^53 - 1)) * 2^-53                                        [uniform_real_distribution<double>]
 *   multinomial(probs, 1): q_k = (float)(-log1p(-uniform)) for k = 0..K-1, argmax_k of probs_k / q_k   [the n_sample == 1 fast path]
 *   normal      Box-Muller on doubles: u1, u2 uniform; r = sqrt(-2 log1p(-u2)), theta = 2 pi u1; returns r cos(theta) and CACHES
 *               r sin(theta) for the next call (the cache lives in the generator, reset by manual_seed)   [normal_distribution<double>]
 *   torch.normal(mean, std) over K elements = (float) normal, then * std + mean. */
static uint32_t tmt_next(rng_t* g) {
    uint32_t* mt = g->tmt;
    if (g->tmti >= 624) {
        int kk;
        uint32_t y;
        for (kk = 0; kk < 624 - 397; ++kk) { y = (mt[kk] & 0x80000000u) | (mt[kk + 1] & 0x7fffffffu); mt[kk] = mt[kk + 397] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u); }
        for (; kk < 623; ++kk) { y = (mt[kk] & 0x80000000u) | (mt[kk + 1] & 0x7fffffffu); mt[kk] = mt[kk + (397 - 624)] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u); }
        y = (mt[623] & 0x80000000u) | (mt[0] & 0x7fffffffu);
        mt[623] = mt[396] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
        g->tmti = 0;
    }
    uint32_t y = mt[g->tmti++];
    y ^= y >> 11; y ^= (y << 7) & 0x9d2c5680u; y ^= (y << 15) & 0xefc60000u; y ^= y >> 18;
    g->tdraws++;
    return y;
}
static void torch_manual_seed(rng_t* g, uint64_t seed) {
    mt_init_genrand(g->tmt, (uint32_t)seed);
    g->tmti = 624; g->tcache_valid = 0; g->tcache = 0.0; g->tdraws = 0;
}
static double torch_uniform(rng_t* g) {
    const uint64_t hi = tmt_next(g), lo = tmt_next(g);
    return (double)(((hi << 32) | lo) & ((1ULL << 53) - 1)) * (1.0 / 9007199254740992.0);
}
static double torch_neglog1m(const azo_config* c, double u) { /* -log1p(-u); 1 - u is exact for a 53-bit u */
    return c->math_mode == AZO_MATH_DET ? -azo_det_log(1.0 - u) : -log1p(-u);
}
static double torch_normal(const azo_config* c, rng_t* g) {
    if (g->tcache_valid) { g->tcache_valid = 0; return g->tcache; }
    const double u1 = torch_uniform(g), u2 = torch_uniform(g);
    const double r = sqrt(2.0 * torch_neglog1m(c, u2)), th = 6.283185307179586 * u1;
    g->tcache = r * (c->math_mode == AZO_MATH_DET ? azo_det_sin(th) : sin(th));
    g->tcache_valid = 1;
    return r * (c->math_mode == AZO_MATH_DET ? azo_det_cos(th) : cos(th));
}
static float torch_sample_action(const azo_config* c, const float* head, rng_t* g) {
    const int K = c->num_components;
    int k = 0;
    if (K > 1) {
        float best = 0.0f;
        for (int i = 0; i < K; ++i) {
            const float q = (float)torch_neglog1m(c, torch_uniform(g));
            const float w = head[2 * K + i] / q;
            if (i == 0 || w > best) { best = w; k = i; }
        }
    }
    float z = 0.0f;
    for (int i = 0; i < K; ++i) {
        const float zi = (float)torch_normal(c, g);
        if (i == k) z = zi;
    }
    float x = z * head[K + k] + head[k];
    float t = c->math_mode == AZO_MATH_DET ? azo_det_tanhf(x) : tanhf(x);
    return c->action_bound > 0.0f ? c->action_bound * t : x;
}

/* random.random() */
static double rng_random(rng_t* g) {
    if (!g->mt_mode) return (double)u32_to_unit(rng_next(g));
    const uint32_t a = mt_next(g) >> 5, b = mt_next(g) >> 6;
    return ((double)a * 67108864.0 + (double)b) * (1.0 / 9007199254740992.0);
}
/* random.choice over n items / random.randint(0, n - 1) */
static int rng_below(rng_t* g, int n) {
    if (!g->mt_mode) return u32_to_index(rng_next(g), n);
    int k = 0;
    while ((n >> k) != 0) ++k; /* n.bit_length() */
    uint32_t r = mt_next(g) >> (32 - k);
    while ((int)r >= n) r = mt_next(g) >> (32 - k);
    return (int)r;
}

/* helpers.py:30-52: winners = where(x == max(x)); random.choice(winners) -- one draw even for one winner */
static int argmax_tiebreak(const double* x, int n, rng_t* g, int* err) {
    double m = x[0];
    int nan = x[0] != x[0];
    for (int i = 1; i < n; ++i) { if (x[i] != x[i]) nan = 1; if (x[i] > m) m = x[i]; }
    if (nan) { *err = -3; return 0; }
    int nw = 0;
    for (int i = 0; i < n; ++i) nw += (x[i] == m);
    int pick = rng_below(g, nw);
    for (int i = 0; i < n; ++i) if (x[i] == m && pick-- == 0) return i;
    return 0;
}

/* mcts.py:488-493 / :736-741 + epsilon_greedy :175-195 */
static int select_index(const azo_config* c, const double* uct, int n, rng_t* g, int* err) {
    if (c->epsilon == 0) return argmax_tiebreak(uct, n, g, err);
    double u = rng_random(g);
    if (u < c->epsilon) return rng_below(g, n);
    return argmax_tiebreak(uct, n, g, err);
}

/* numpy pairwise summation for n <= 128 (np.sum in get_on_policy_value_target, mcts.py:111) */
static double np_sum(const double* a, int n) {
    if (n < 8) { double r = 0.; for (int i = 0; i < n; ++i) r += a[i]; return r; }
    double r[8];
    for (int k = 0; k < 8; ++k) r[k] = a[k];
    int i;
    for (i = 8; i < n - (n % 8); i += 8) for (int k = 0; k < 8; ++k) r[k] += a[i + k];
    double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; ++i) res += a[i];
    return res;
}

static double value_target(const azo_config* c, const double* Q, const int32_t* counts, int n) {
    if (c->v_target == AZO_VT_ON_POLICY) {
        double tmp[256];
        int64_t tot = 0;
        for (int i = 0; i < n; ++i) tot += counts[i];
        for (int i = 0; i < n; ++i) tmp[i] = ((double)counts[i] / (double)tot) * Q[i];
        return np_sum(tmp, n);
    }
    /* off_policy (mcts.py:131) and greedy from a non-terminal root (mcts.py:155 never loops): Q.max() */
    double m = Q[0];
    for (int i = 1; i < n; ++i) m = Q[i] > m ? Q[i] : m;
    return m;
}

/* ------------------------------------------------------------------------------------------------
 * Discrete search (mcts.py:418-462).
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    int R, A;
    int n_nodes;
    int32_t *parent, *paction, *node_n, *terminal, *en, *echild;
    float *V, *prior;
    double *r, *state, *eW;
} dtree_t;

static void dtree_alloc(dtree_t* t, int R, int A) {
    t->R = R; t->A = A;
    t->parent = calloc(R, 4); t->paction = calloc(R, 4); t->node_n = calloc(R, 4); t->terminal = calloc(R, 4);
    t->en = calloc((size_t)R * A, 4); t->echild = calloc((size_t)R * A, 4);
    t->V = calloc(R, 4); t->prior = calloc((size_t)R * A, 4);
    t->r = calloc(R, 8); t->state = calloc((size_t)R * 4, 8); t->eW = calloc((size_t)R * A, 8);
}
static void dtree_clear(dtree_t* t) {
    const size_t R = t->R, A = t->A;
    memset(t->parent, 0, R * 4); memset(t->paction, 0, R * 4); memset(t->node_n, 0, R * 4); memset(t->terminal, 0, R * 4);
    memset(t->en, 0, R * A * 4); memset(t->echild, 0, R * A * 4); memset(t->V, 0, R * 4); memset(t->prior, 0, R * A * 4);
    memset(t->r, 0, R * 8); memset(t->state, 0, R * 4 * 8); memset(t->eW, 0, R * A * 8);
}
static void dtree_free(dtree_t* t) {
    free(t->parent); free(t->paction); free(t->node_n); free(t->terminal); free(t->en); free(t->echild);
    free(t->V); free(t->prior); free(t->r); free(t->state); free(t->eW);
}

/* mcts.py:385-416 */
static void d_evaluate(const azo_config* c, const net_t* net, const azo_tapes* tp, int64_t b, dtree_t* t, int node, int64_t* ctr) {
    const int A = t->A;
    float V, raw[AZO_MAX_A];
    if (c->use_eval_tape) {
        V = tp->V[b * t->R + node];
        for (int a = 0; a < A; ++a) t->prior[node * A + a] = tp->prior[(b * t->R + node) * A + a];
    } else {
        float x[ENV_MAX_OBS];
        env_obs(c, t->state + node * 4, x);
        net_forward(net, c, x, &V, raw);
        azo_head_post(c, raw, t->prior + node * A);
        ctr[4]++;
    }
    t->V[node] = t->terminal[node] ? 0.0f : V;
    for (int a = 0; a < A; ++a) { t->eW[node * A + a] = 0.0; t->en[node * A + a] = 0; t->echild[node * A + a] = -1; }
}

static int search_discrete_one(const azo_config* c, const net_t* net, const azo_tapes* tp, int64_t b, const double* root_state,
                               int32_t root_n, dtree_t* t, rng_t* g, int64_t* ctr) {
    const int A = t->A;
    int err = 0;
    dtree_clear(t);
    t->n_nodes = 1;
    t->parent[0] = -1; t->paction[0] = -1; t->node_n[0] = root_n; t->terminal[0] = 0; t->r[0] = 0.0;
    for (int i = 0; i < env_hidden_dim(c); ++i) t->state[i] = root_state[i];
    d_evaluate(c, net, tp, b, t, 0, ctr);
    for (int it = 0; it < c->n_rollouts; ++it) {
        int node = 0, created = 0;
        while (!t->terminal[node]) {
            double uct[AZO_MAX_A];
            double sq = sqrt((double)(t->node_n[node] + 1));
            for (int a = 0; a < A; ++a) {
                int n = t->en[node * A + a];
                double Q = n > 0 ? t->eW[node * A + a] / (double)n : (double)t->V[node];
                double pc = c->puct_f32 ? (double)(t->prior[node * A + a] * (float)c->c_uct) : (double)t->prior[node * A + a] * c->c_uct;
                uct[a] = Q + pc * (sq / (double)(n + 1)); /* mcts.py:483-484 */
            }
            int a = select_index(c, uct, A, g, &err);
            if (err) return err;
            ctr[1]++; ctr[2] += A;
            int child = t->echild[node * A + a];
            if (child >= 0) { node = child; continue; }
            child = t->n_nodes++;
            double rew;
            int term = env_step(c, t->state + node * 4, (float)a, t->state + child * 4, &rew);
            if (term == AZO_ERR_WRAP) return AZO_ERR_WRAP;
            /* CartPole's reward wrappers (rl/wrappers.py): a constant per terminal flag; azo_search allows 1.0 / 1.0 only on other envs */
            if (c->reward_step != 1.0 || c->reward_terminal != 1.0) rew = term ? c->reward_terminal : c->reward_step;
            t->parent[child] = node; t->paction[child] = a; t->node_n[child] = 0; t->terminal[child] = term; t->r[child] = rew;
            t->echild[node * A + a] = child;
            d_evaluate(c, net, tp, b, t, child, ctr);
            node = child;
            created = 1;
            break;
        }
        if (!created) ctr[6]++; /* trace ended on an already existing terminal node */
        /* mcts.py:241-267 */
        double R = (double)t->V[node];
        while (t->parent[node] >= 0) {
            R = t->r[node] + c->gamma * R;
            int p = t->parent[node], a = t->paction[node];
            t->en[p * A + a] += 1;
            t->eW[p * A + a] += R;
            node = p;
            t->node_n[node] += 1;
        }
        ctr[0]++;
    }
    return 0;
}

/* ------------------------------------------------------------------------------------------------
 * Continuous search with progressive widening (mcts.py:656-741).
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    int R, K3;
    int n_rows;
    int32_t *parent, *en, *expanded, *node_n, *terminal;
    float *action, *V, *head;
    double *eW, *r, *state;
} ctree_t;

static void ctree_alloc(ctree_t* t, int R, int K3) {
    t->R = R; t->K3 = K3;
    t->parent = calloc(R, 4); t->en = calloc(R, 4); t->expanded = calloc(R, 4); t->node_n = calloc(R, 4); t->terminal = calloc(R, 4);
    t->action = calloc(R, 4); t->V = calloc(R, 4); t->head = calloc((size_t)R * K3, 4);
    t->eW = calloc(R, 8); t->r = calloc(R, 8); t->state = calloc((size_t)R * 2, 8);
}
static void ctree_clear(ctree_t* t) {
    const size_t R = t->R;
    memset(t->parent, 0, R * 4); memset(t->en, 0, R * 4); memset(t->expanded, 0, R * 4); memset(t->node_n, 0, R * 4);
    memset(t->terminal, 0, R * 4); memset(t->action, 0, R * 4); memset(t->V, 0, R * 4); memset(t->head, 0, R * t->K3 * 4);
    memset(t->eW, 0, R * 8); memset(t->r, 0, R * 8); memset(t->state, 0, R * 2 * 8);
}
static void ctree_free(ctree_t* t) {
    free(t->parent); free(t->en); free(t->expanded); free(t->node_n); free(t->terminal);
    free(t->action); free(t->V); free(t->head); free(t->eW); free(t->r); free(t->state);
}

/* add_value_estimate (mcts.py:602-623); also caches the policy head of the node, which the reference
 * recomputes on every add_pw_action (mcts.py:631-635 notes it is deterministic given the state). */
static void c_evaluate(const azo_config* c, const net_t* net, const azo_tapes* tp, int64_t b, ctree_t* t, int row, int64_t* ctr) {
    float V;
    if (c->use_eval_tape) {
        V = tp->V[b * t->R + row];
    } else {
        float obs[ENV_MAX_OBS], raw[3 * AZO_MAX_K];
        env_obs(c, t->state + row * 2, obs);
        net_forward(net, c, obs, &V, raw);
        azo_head_post(c, raw, t->head + (size_t)row * t->K3);
        ctr[4]++;
    }
    t->V[row] = t->terminal[row] ? 0.0f : V;
}

/* add_pw_action (mcts.py:625-654) */
static int c_add_pw_action(const azo_config* c, const azo_tapes* tp, int64_t b, ctree_t* t, int node, rng_t* g, int64_t* ctr) {
    int row = t->n_rows++;
    float a;
    if (c->use_eval_tape) {
        a = tp->action[b * t->R + row];
        g->pw++;
    } else {
        if (g->mt_mode) {
            a = torch_sample_action(c, t->head + (size_t)node * t->K3, g);
            g->pw++;
        } else {
            float u, z[AZO_MAX_K];
            azo_noise(g->seed, g->tree, g->pw++, c->num_components, &u, z);
            a = azo_sample_action(c, t->head + (size_t)node * t->K3, u, z);
        }
    }
    t->parent[row] = node; t->action[row] = a; t->eW[row] = 0.0; t->en[row] = 0; t->expanded[row] = 0;
    t->node_n[row] = 0; t->terminal[row] = 0; t->V[row] = 0.0f; t->r[row] = 0.0;
    ctr[3]++;
    return row;
}

static int search_continuous_one(const azo_config* c, const net_t* net, const azo_tapes* tp, int64_t b, const double* root_state,
                                 ctree_t* t, rng_t* g, const int32_t* pw_table, int64_t* ctr) {
    int err = 0;
    int path[4096];
    ctree_clear(t);
    t->n_rows = 1;
    t->parent[0] = -1; t->expanded[0] = 1; t->node_n[0] = 0; t->terminal[0] = 0; t->r[0] = 0.0; t->en[0] = 0; t->eW[0] = 0.0;
    t->action[0] = 0.0f;
    for (int i = 0; i < env_hidden_dim(c); ++i) t->state[i] = root_state[i];
    c_evaluate(c, net, tp, b, t, 0, ctr);
    c_add_pw_action(c, tp, b, t, 0, g, ctr);
    const float g32 = (float)c->gamma;
    for (int it = 0; it < c->n_rollouts; ++it) {
        int node = 0, depth = 0, created = 0;
        while (!t->terminal[node]) {
            int kids[4096], C = 0;
            for (int i = 1; i < t->n_rows; ++i) if (t->parent[i] == node) kids[C++] = i;
            int sel;
            if (pw_table[t->node_n[node]] - C > 0) { /* states.py:252-275 */
                sel = c_add_pw_action(c, tp, b, t, node, g, ctr);
            } else {
                double uct[4096];
                double sq = sqrt((double)(t->node_n[node] + 1));
                for (int j = 0; j < C; ++j) {
                    int n = t->en[kids[j]];
                    double Q = n > 0 ? t->eW[kids[j]] / (double)n : (double)t->V[node];
                    uct[j] = Q + c->c_uct * (sq / (double)(n + 1)); /* mcts.py:731-732 */
                }
                sel = kids[select_index(c, uct, C, g, &err)];
                if (err) return err;
                ctr[2] += C;
            }
            ctr[1]++;
            path[depth++] = sel;
            if (t->expanded[sel]) { node = sel; continue; }
            double rew;
            int term = env_step(c, t->state + node * 2, t->action[sel], t->state + sel * 2, &rew);
            t->r[sel] = rew / PENDULUM_R_SCALE; /* mcts.py:687 */
            t->terminal[sel] = term; t->expanded[sel] = 1; t->node_n[sel] = 0;
            c_evaluate(c, net, tp, b, t, sel, ctr);
            node = sel;
            created = 1;
            break;
        }
        if (!created) ctr[6]++;
        /* backprop (mcts.py:241-267).  First step: gamma * (0-d f32 array) stays f32 under NEP 50. */
        double R = 0.0;
        for (int d = depth - 1; d >= 0; --d) {
            int row = path[d];
            if (d == depth - 1) R = t->r[row] + (double)(g32 * t->V[row]);
            else R = t->r[row] + c->gamma * R;
            t->en[row] += 1;
            t->eW[row] += R;
            t->node_n[t->parent[row]] += 1;
        }
        ctr[0]++;
    }
    return 0;
}

/* ------------------------------------------------------------------------------------------------
 * Batch driver (pthreads; trees are independent, so results do not depend on the thread count).
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    const azo_config* cfg; const net_t* net; const azo_tapes* tapes; const double* root_state; const int32_t* root_n_init;
    int64_t tree_id0; int32_t B; azo_results* res; azo_dump_discrete* dd; azo_dump_continuous* dc; const int32_t* pw_table;
    int64_t* next; int* rc; int64_t ctr[8];
} job_t;

static void* worker(void* arg) {
    job_t* J = (job_t*)arg;
    const azo_config* cfg = J->cfg;
    const int R = azo_rows(cfg);
    const int A = cfg->num_actions, K = cfg->num_components, K3 = 3 * (K > 0 ? K : 1), HS = env_hidden_dim(cfg);
    azo_results* res = J->res;
    dtree_t dt; ctree_t ct;
    if (cfg->variant == AZO_DISCRETE) dtree_alloc(&dt, R, A); else ctree_alloc(&ct, R, K3);
    for (;;) {
        int64_t b0 = __atomic_fetch_add(J->next, 16, __ATOMIC_RELAXED);
        if (b0 >= J->B) break;
        int64_t b1 = b0 + 16 < J->B ? b0 + 16 : J->B;
        for (int64_t b = b0; b < b1; ++b) {
            rng_t g;
            g.seed = cfg->seed; g.tree = J->tree_id0 + b; g.draws = 0; g.pw = 0; g.mt_mode = cfg->rng_mode == 1; g.mti = 624;
            if (g.mt_mode) {
                mt_seed(&g, cfg->seed + (uint64_t)(J->tree_id0 + b));
                torch_manual_seed(&g, cfg->seed + (uint64_t)(J->tree_id0 + b));
            }
            int e;
            if (cfg->variant == AZO_DISCRETE) {
                e = search_discrete_one(cfg, J->net, J->tapes, b, J->root_state + b * HS, J->root_n_init ? J->root_n_init[b] : 0, &dt, &g, J->ctr);
                if (!e && res) {
                    double Q[AZO_MAX_A] = {0};
                    res->n_children[b] = A;
                    for (int a = 0; a < A; ++a) {
                        int n = dt.en[a];
                        Q[a] = n > 0 ? dt.eW[a] / (double)n : (double)dt.V[0];
                        res->actions[b * res->cmax + a] = (float)a;
                        res->counts[b * res->cmax + a] = n;
                        res->Q[b * res->cmax + a] = Q[a];
                    }
                    res->V_target[b] = value_target(cfg, Q, dt.en, A);
                }
                if (!e && J->dd) {
                    azo_dump_discrete* dd = J->dd;
                    dd->n_nodes[b] = dt.n_nodes;
                    size_t o = (size_t)b * R;
                    memcpy(dd->parent + o, dt.parent, R * 4); memcpy(dd->paction + o, dt.paction, R * 4);
                    memcpy(dd->node_n + o, dt.node_n, R * 4); memcpy(dd->terminal + o, dt.terminal, R * 4);
                    memcpy(dd->V + o, dt.V, R * 4); memcpy(dd->r + o, dt.r, R * 8);
                    for (int i = 0; i < R; ++i) memcpy(dd->state + (o + i) * HS, dt.state + (size_t)i * 4, (size_t)HS * 8);
                    memcpy(dd->prior + o * A, dt.prior, (size_t)R * A * 4); memcpy(dd->eW + o * A, dt.eW, (size_t)R * A * 8);
                    memcpy(dd->en + o * A, dt.en, (size_t)R * A * 4); memcpy(dd->echild + o * A, dt.echild, (size_t)R * A * 4);
                }
            } else {
                e = search_continuous_one(cfg, J->net, J->tapes, b, J->root_state + b * HS, &ct, &g, J->pw_table, J->ctr);
                if (!e && res) {
                    double Q[4096]; int32_t cnt[4096]; int C = 0;
                    Q[0] = 0.0;
                    for (int i = 1; i < ct.n_rows; ++i) if (ct.parent[i] == 0 && C < res->cmax) {
                        int n = ct.en[i];
                        Q[C] = n > 0 ? ct.eW[i] / (double)n : (double)ct.V[0];
                        cnt[C] = n;
                        res->actions[b * res->cmax + C] = ct.action[i];
                        res->counts[b * res->cmax + C] = n;
                        res->Q[b * res->cmax + C] = Q[C];
                        ++C;
                    }
                    res->n_children[b] = C;
                    res->V_target[b] = value_target(cfg, Q, cnt, C);
                }
                if (!e && J->dc) {
                    azo_dump_continuous* dc = J->dc;
                    dc->n_rows[b] = ct.n_rows;
                    size_t o = (size_t)b * R;
                    memcpy(dc->parent + o, ct.parent, R * 4); memcpy(dc->action + o, ct.action, R * 4);
                    memcpy(dc->eW + o, ct.eW, R * 8); memcpy(dc->en + o, ct.en, R * 4);
                    memcpy(dc->expanded + o, ct.expanded, R * 4); memcpy(dc->node_n + o, ct.node_n, R * 4);
                    memcpy(dc->terminal + o, ct.terminal, R * 4); memcpy(dc->V + o, ct.V, R * 4);
                    memcpy(dc->r + o, ct.r, R * 8); memcpy(dc->state + o * 2, ct.state, (size_t)R * 2 * 8);
                    memcpy(dc->head + o * K3, ct.head, (size_t)R * K3 * 4);
                }
            }
            J->ctr[5] += g.draws;
            if (e) __atomic_store_n(J->rc, e, __ATOMIC_RELAXED);
        }
    }
    if (cfg->variant == AZO_DISCRETE) dtree_free(&dt); else ctree_free(&ct);
    return NULL;
}

int azo_search(const azo_config* cfg, const float* weights, int64_t n_weights, int32_t B, const double* root_state,
               const int32_t* root_n_init, int64_t tree_id0, const azo_tapes* tapes, azo_results* res,
               azo_dump_discrete* dd, azo_dump_continuous* dc, int32_t n_threads) {
    const int R = azo_rows(cfg);
    if (R > 4096 || cfg->hidden > 1024) return -2;
    if (cfg->variant == AZO_DISCRETE && (cfg->num_actions < 1 || cfg->num_actions > AZO_MAX_A)) return -2;
    if (cfg->variant == AZO_CONTINUOUS && (cfg->num_components < 1 || cfg->num_components > AZO_MAX_K)) return -2;
    if (cfg->use_eval_tape && !tapes) return -2;
    const int disc = cfg->variant == AZO_DISCRETE, S = cfg->state_dim, A = cfg->num_actions;
    if (cfg->env == AZO_ENV_MOUNTAIN_CAR_CONTINUOUS && !(!disc && S == 2)) return -2;
    if (cfg->env == AZO_ENV_MOUNTAIN_CAR && !(disc && A == 3 && S == 2)) return -2;
    if (cfg->env == AZO_ENV_ACROBOT && !(disc && A == 3 && S == 6)) return -2;
    if (cfg->env < AZO_ENV_DEFAULT || cfg->env > AZO_ENV_ACROBOT) return -2;
    if (!(disc && cfg->env == AZO_ENV_DEFAULT) && (cfg->reward_step != 1.0 || cfg->reward_terminal != 1.0)) return -2;
    net_t net;
    memset(&net, 0, sizeof net);
    if (!cfg->use_eval_tape && net_init(&net, cfg, weights, n_weights)) return -2;
    int32_t* pw_table = NULL;
    if (cfg->variant == AZO_CONTINUOUS) {
        pw_table = malloc(sizeof(int32_t) * (cfg->n_rollouts + 2));
        for (int n = 0; n < cfg->n_rollouts + 2; ++n) pw_table[n] = azo_pw_limit(cfg->c_pw, cfg->kappa, n);
    }
    int rc = 0;
    int64_t next = 0;
    if (n_threads < 1) n_threads = 1;
    if (n_threads > 256) n_threads = 256;
    job_t jobs[256];
    pthread_t th[256];
    for (int i = 0; i < n_threads; ++i) {
        job_t j = {cfg, &net, tapes, root_state, root_n_init, tree_id0, B, res, dd, dc, pw_table, &next, &rc, {0}};
        jobs[i] = j;
    }
    for (int i = 1; i < n_threads; ++i) pthread_create(&th[i], NULL, worker, &jobs[i]);
    worker(&jobs[0]);
    for (int i = 1; i < n_threads; ++i) pthread_join(th[i], NULL);
    if (res && res->counters) {
        for (int k = 0; k < 8; ++k) res->counters[k] = 0;
        for (int i = 0; i < n_threads; ++i) for (int k = 0; k < 8; ++k) res->counters[k] += jobs[i].ctr[k];
    }
    free(pw_table);
    if (!cfg->use_eval_tape) net_free(&net);
    return rc;
}

/* ------------------------------------------------------------------------------------------------
 * Building blocks for the primitive tests (azg_oracle.h): batched deterministic functions, and the
 * MT19937 generators on a caller-held state.
 * ---------------------------------------------------------------------------------------------- */
typedef struct { int32_t fn; const void* in; void* out; int64_t i0, i1; } eval_job_t;

static void* eval_worker(void* arg) {
    const eval_job_t* J = (const eval_job_t*)arg;
    const float* fi = (const float*)J->in; float* fo = (float*)J->out;
    const double* di = (const double*)J->in; double* dout = (double*)J->out;
    azo_config c;
    memset(&c, 0, sizeof c);
    c.math_mode = AZO_MATH_DET;
    c.activation = J->fn - AZO_FN_ACT;
    for (int64_t i = J->i0; i < J->i1; ++i) {
        switch (J->fn) {
            case AZO_FN_EXPF: fo[i] = azo_det_expf(fi[i]); break;
            case AZO_FN_EXPM1F: fo[i] = azo_det_expm1f(fi[i]); break;
            case AZO_FN_TANHF: fo[i] = azo_det_tanhf(fi[i]); break;
            case AZO_FN_SIN: dout[i] = azo_det_sin(di[i]); break;
            case AZO_FN_COS: dout[i] = azo_det_cos(di[i]); break;
            case AZO_FN_LOG: dout[i] = azo_det_log(di[i]); break;
            default: fo[i] = act_fn(&c, fi[i]); break;
        }
    }
    return NULL;
}

int azo_det_eval(int32_t fn, const void* in, void* out, int64_t n, int32_t n_threads) {
    if (!((fn >= AZO_FN_EXPF && fn <= AZO_FN_LOG) || (fn >= AZO_FN_ACT && fn <= AZO_FN_ACT + AZO_ACT_HARDSWISH))) return -2;
    if (n_threads < 1) n_threads = 1;
    if (n_threads > 256) n_threads = 256;
    eval_job_t jobs[256];
    pthread_t th[256];
    for (int i = 0; i < n_threads; ++i) {
        eval_job_t j = {fn, in, out, n * i / n_threads, n * (i + 1) / n_threads};
        jobs[i] = j;
    }
    for (int i = 1; i < n_threads; ++i) pthread_create(&th[i], NULL, eval_worker, &jobs[i]);
    eval_worker(&jobs[0]);
    for (int i = 1; i < n_threads; ++i) pthread_join(th[i], NULL);
    return 0;
}

/* st = 624 state words + the index word; the generators of rng_t run on a copy */
static void mt_load(rng_t* g, const uint32_t* st) { memcpy(g->mt, st, 624 * 4); g->mti = (int)st[624]; g->draws = 0; }
static void mt_store(const rng_t* g, uint32_t* st) { memcpy(st, g->mt, 624 * 4); st[624] = (uint32_t)g->mti; }

void azo_mt_seed(uint32_t* st, uint64_t seed) { rng_t g; mt_seed(&g, seed); mt_store(&g, st); }
uint32_t azo_mt_u32(uint32_t* st) { rng_t g; mt_load(&g, st); const uint32_t r = mt_next(&g); mt_store(&g, st); return r; }
double azo_mt_random(uint32_t* st) {
    rng_t g; mt_load(&g, st); g.mt_mode = 1;
    const double r = rng_random(&g);
    mt_store(&g, st);
    return r;
}
int32_t azo_mt_below(uint32_t* st, int32_t n) {
    rng_t g; mt_load(&g, st); g.mt_mode = 1;
    const int32_t r = rng_below(&g, n);
    mt_store(&g, st);
    return r;
}
void azo_torch_seed(uint32_t* st, uint64_t seed) { rng_t g; torch_manual_seed(&g, seed); memcpy(st, g.tmt, 624 * 4); st[624] = (uint32_t)g.tmti; }
double azo_torch_uniform(uint32_t* st) {
    rng_t g; memcpy(g.tmt, st, 624 * 4); g.tmti = (int)st[624]; g.tdraws = 0;
    const double r = torch_uniform(&g);
    memcpy(st, g.tmt, 624 * 4); st[624] = (uint32_t)g.tmti;
    return r;
}

void azo_rng_block_batch(uint64_t seed, const int64_t* tree, const int32_t* stream, const int64_t* idx, const int32_t* block, int64_t n,
                         uint32_t* out) {
    for (int64_t i = 0; i < n; ++i) rng_block(seed, tree[i], stream[i], idx[i], block[i], out + 4 * i);
}

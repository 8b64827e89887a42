"""An f64 evaluation of the policy network with a derived bound on the error of the engine's evaluation contracts.

`forward(cfg, w, x)` evaluates the flat weight vector (network.py layout: trunk layers, value head, dist head) in f64 and, next to
every value, a bound E such that the FP32 contract (AZO_EVAL_FP32, csrc/mlp.cuh) and the Q8 contract (AZO_EVAL_Q8,
oracle/azg_oracle.h; csrc/qmlp2.cuh, csrc/search_wg.cuh) both land within E of it.  The bound is carried through the layers.
u = 2^-24 is the unit roundoff of f32, gamma_n = n u / (1 - n u).

Notation for one layer: a is the exact (f64) input, e >= |a_hat - a| the bound on the computed input, y = b + W a the exact
output, y_hat the computed one.

* FP32 layer (every layer of the FP32 contract; layer 0 of Q8): acc_0 = b, acc_k = fma(w_k, a_hat_k, acc_{k-1}), k ascending.
  Each fma rounds once, so |y_hat - (b + W a_hat)| <= u sum_k |acc_k| (1 + 2 gamma_K), and |acc_k| <= |s_k| + c_k with s_k the
  exact partial sums and c_k = sum_{i<=k} |w_i| e_i.  With |W (a_hat - a)| <= |W| e:
      |y_hat - y| <= |W| e + u (1 + 2 gamma_K) sum_k (|s_k| + c_k).
* Q8 hidden layer (l >= 1).  Activations of a row are scaled by 2^(149 - ex), ex = clamp(biased exponent of f32(vmax 1.004f),
  32, 200), and rounded to integers; one unit is ux = 2^(ex - 149), the rounding moves each input by at most ux / 2.  ex depends
  on the computed vmax, which lies in [vmax - max e, vmax + max e]: the bound takes the largest exponent of that range.  Weights
  of output j are scaled the same way with their own exponent ew_j (unit uw_j); their rounding eta = w_q - w is known exactly,
  so it enters with its sign: |sum_k eta_k a_k| + sum_k |eta_k| e_k.  The integer products are exact; the contract keeps the
  digit products of order 4 and higher (PA, PB, PC) and drops D = 2^8 (xm wl + xl wm) + xl wl, with |xm|, |xl| <= 128 and the
  weight digits wm, wl known: |D| ux uw_j <= ux uw_j sum_k (2^15 (|wl_k| + |wm_k|) + 2^7 |wl_k|).  The f32 recombination
  fma(fma(PA, 256, PB), 256, PC) rounds twice; in real units its two intermediates are bounded by M = sum_k |w_q,k| (|a_k| + e_k
  + ux / 2) plus |D| and the PC part, 2^16 ux uw_j 2^7 sum_k (|wh_k| + |wm_k| + |wl_k|), so it adds at most 2 u (1 + u) that sum.
  The scale cx cw_j = 2^(ex + ew_j - 282) is exact while it is a normal f32; below 2^-126 it is rounded (or flushed), which
  moves the product by at most M 2^-150 / (cx cw_j) (and never by more than M).  The final fma with the bias rounds once: u |y_hat|.
* Heads in Q8: partial sums of 32 products each start from 0, are added pairwise and then to the bias: the same running bound
  over every partial sum, every pairwise sum and the final sum.
* Activations: relu, elu, leaky relu and relu6 are 1-Lipschitz, silu is 1.1-Lipschitz, hardswish 1.5-Lipschitz; computing the
  activation itself (deterministic expm1f / expf, one or two roundings) adds at most 8 u (|act(y)| + |y|).
* Head post-processing.  Softmax: logits that each move by at most eps move every probability by a factor within
  [e^(-2 eps), e^(2 eps)]; computing it (x - max, det expf, a sum of n terms, a division) adds a relative
  2 u |x - max| + (n + 8) u.  sigma = exp(clamp(log sigma)): clamp is 1-Lipschitz, so the relative error is e^eps - 1 + 4 u.
  mu is the raw output.

`q8_contract` restates the Q8 contract in numpy (f32 fma emulated in f64), layer by layer, so that tests can show the bound
rejects a contract that is subtly wrong.
"""
from __future__ import annotations

import numpy as np

from oracle import azo

U = 2.0 ** -24
LIPSCHITZ = {azo.ACT_RELU: 1.0, azo.ACT_ELU: 1.0, azo.ACT_LEAKYRELU: 1.0, azo.ACT_RELU6: 1.0, azo.ACT_SILU: 1.1,
             azo.ACT_HARDSWISH: 1.5}


def gamma(n: int) -> float:
    return n * U / (1 - n * U)


def split(cfg: azo.Config, w: np.ndarray):
    """Flat weights -> [(W [H, K], b [H])] per trunk layer, value head (wv [H], bv), dist head (wd [P, H], bd [P])."""
    H, S, L, P = cfg.hidden, cfg.state_dim, cfg.n_hidden, cfg.head_dim
    w = np.asarray(w, np.float32)
    assert w.size == cfg.num_weights
    layers, o = [], 0
    for l in range(L):
        K = S if l == 0 else H
        layers.append((w[o:o + H * K].reshape(H, K), w[o + H * K:o + H * K + H]))
        o += H * K + H
    wv, bv = w[o:o + H], w[o + H]
    o += H + 1
    wd, bd = w[o:o + P * H].reshape(P, H), w[o + P * H:o + P * H + P]
    return layers, (wv, bv), (wd, bd)


def act64(act: int, v: np.ndarray) -> np.ndarray:
    if act == azo.ACT_RELU:
        return np.maximum(v, 0.0)
    if act == azo.ACT_ELU:
        return np.where(v > 0, v, np.expm1(np.minimum(v, 0.0)))
    if act == azo.ACT_LEAKYRELU:
        return np.where(v > 0, v, 0.01 * v)
    if act == azo.ACT_RELU6:
        return np.clip(v, 0.0, 6.0)
    if act == azo.ACT_SILU:
        return v / (1.0 + np.exp(-np.clip(v, -700, 700)))
    return v * np.clip(v + 3.0, 0.0, 6.0) / 6.0


def biased_exponent(v: np.ndarray) -> np.ndarray:
    """Biased f32 exponent of positive f64 values, clamped to [32, 200] as the contract clamps it (0 -> 32)."""
    v = np.asarray(v, np.float64)
    e = np.frexp(np.where(v > 0, v, 1.0))[1].astype(np.int64) - 1 + 127  # frexp: v = m 2^E, m in [0.5, 1)
    return np.clip(np.where(v > 0, e, 32), 32, 200)


def quantise_weights(W: np.ndarray):
    """Exact Q8 weight quantisation of one hidden layer (engine.cu pack_weights_q8): integer weights, per-output unit uw, and the
    three balanced base-256 digits."""
    W = np.asarray(W, np.float32)
    wmax = np.abs(W).max(axis=1)
    ew = biased_exponent((wmax * np.float32(1.004)).astype(np.float32).astype(np.float64))
    uw = np.ldexp(1.0, ew - 149)
    q = np.rint(W.astype(np.float64) / uw[:, None]).astype(np.int64)
    t = (q + 0x8080) ^ 0x8080
    dig = [((t >> s) & 0xFF).astype(np.int64) for s in (16, 8, 0)]
    dig = [np.where(d > 127, d - 256, d) for d in dig]
    return q, uw, ew, dig


def _fp32_layer(W, b, a, e):
    """Running bound of one f32 FMA chain (from the bias, k ascending) per output; a, e: [n, K]."""
    W64, b64 = W.astype(np.float64), b.astype(np.float64)
    terms = a[:, None, :] * W64[None, :, :]                       # [n, H, K]
    s = b64[None, :, None] + np.cumsum(terms, axis=2)
    c = np.cumsum(np.abs(W64)[None, :, :] * e[:, None, :], axis=2)
    K = W.shape[1]
    y = s[:, :, -1]
    err = c[:, :, -1] + U * (1 + 2 * gamma(K)) * (np.abs(s) + c).sum(axis=2)
    return y, err


def _q8_head(W, b, a, e):
    """Running bound of the Q8 head: 32-term FMA chains from 0, summed pairwise, plus the bias."""
    W64, b64 = W.astype(np.float64), b.astype(np.float64)
    n, H = a.shape
    terms = a[:, None, :] * W64[None, :, :]
    cterm = e[:, None, :] * np.abs(W64)[None, :, :]
    parts, cparts, run = [], [], 0.0
    for q in range(H // 32):
        s = np.cumsum(terms[:, :, 32 * q:32 * q + 32], axis=2)
        c = np.cumsum(cterm[:, :, 32 * q:32 * q + 32], axis=2)
        run = run + (np.abs(s) + c).sum(axis=2)
        parts.append(s[:, :, -1])
        cparts.append(c[:, :, -1])
    span = 1
    while span < len(parts):
        for q in range(0, len(parts) - span, 2 * span):
            parts[q] = parts[q] + parts[q + span]
            cparts[q] = cparts[q] + cparts[q + span]
            run = run + np.abs(parts[q]) + cparts[q]
        span *= 2
    y = parts[0] + b64
    run = run + np.abs(y) + cparts[0]
    return y, cparts[0] + U * (1 + 2 * gamma(H + 8)) * run


def _q8_hidden(W, b, a, e):
    """Bound of one Q8 hidden layer (module docstring); a, e: [n, H]."""
    q, uw, ew, (wh, wm, wl) = quantise_weights(W)
    W64, b64 = W.astype(np.float64), b.astype(np.float64)
    wq = q * uw[:, None]                                           # exact in f64 (|q| < 2^24)
    eta = wq - W64
    y = b64[None, :] + a @ W64.T
    vmax = (np.abs(a) + e).max(axis=1)
    ex = biased_exponent(vmax * 1.004 * (1 + 2 ** -22))
    ux = np.ldexp(1.0, ex - 149)[:, None]                          # [n, 1]
    M = (np.abs(a) + e + ux / 2) @ np.abs(wq).T                    # [n, H]
    err = e @ np.abs(W64).T                                        # propagated input error
    err = err + np.abs(a @ eta.T) * (1 + 2 ** -40) + e @ np.abs(eta).T
    err = err + (ux / 2) * np.abs(wq).sum(axis=1)[None, :]         # input rounding
    D = ux * uw[None, :] * (2.0 ** 15 * (np.abs(wl) + np.abs(wm)).sum(1) + 2.0 ** 7 * np.abs(wl).sum(1))[None, :]
    PCm = ux * uw[None, :] * 2.0 ** 23 * (np.abs(wh) + np.abs(wm) + np.abs(wl)).sum(1)[None, :]
    err = err + D + 2 * U * (1 + U) * (M + D + PCm)
    scale = np.ldexp(1.0, ex[:, None] + ew[None, :] - 282)
    err = err + np.where(scale < 2.0 ** -126, np.minimum(M, M * 2.0 ** -150 / scale), 0.0)
    err = err + U * (np.abs(y) + err) * (1 + U)
    return y, err


def _activate(act, y, err):
    a = act64(act, y)
    e = LIPSCHITZ[act] * err + 8 * U * (np.abs(a) + np.abs(y) + err)
    return a, e


def _softmax_bound(logits, err):
    z = logits - logits.max(axis=1, keepdims=True)
    p = np.exp(z) / np.exp(z).sum(axis=1, keepdims=True)
    eps = np.minimum(err.max(axis=1, keepdims=True), 100.0)
    n = logits.shape[1]
    rel = np.expm1(2 * eps) + 2 * U * (np.abs(z) + 2 * eps) + (n + 8) * U
    # exp below the normal f32 range is subnormal or flushed to 0: an absolute 2^-125 covers it; no probability moves by more than 1
    return p, np.minimum(p * np.exp(2 * eps) * rel + 2.0 ** -125, 1.0)


def forward(cfg: azo.Config, w: np.ndarray, x: np.ndarray, x_err=None, q8=None, trace=False):
    """f64 forward with error bounds.  Returns dict V, head (raw), post (head_post), and bounds bV, bhead, bpost; with
    trace=True also `layers`: [(a, bound)] per trunk layer.  x_err: bound on the input perturbation (default 0)."""
    q8 = cfg.eval_mode == azo.EVAL_Q8 if q8 is None else q8
    x = np.asarray(x, np.float32).reshape(-1, cfg.state_dim)
    if x.shape[0] > 1024:  # the FP32 running bound holds [rows, H, H] partial sums: evaluate in pieces
        if x_err is not None:
            x_err = np.broadcast_to(np.asarray(x_err, np.float64), x.shape)
        parts = [forward(cfg, w, x[i:i + 1024], None if x_err is None else x_err[i:i + 1024], q8) for i in range(0, x.shape[0], 1024)]
        return {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}
    layers, (wv, bv), (wd, bd) = split(cfg, w)
    a = x.astype(np.float64)
    e = np.zeros_like(a) if x_err is None else np.broadcast_to(np.asarray(x_err, np.float64), a.shape).copy()
    trace_out = []
    for l, (W, b) in enumerate(layers):
        y, err = (_q8_hidden if q8 and l > 0 else _fp32_layer)(W, b, a, e)
        a, e = _activate(cfg.activation, y, err)
        trace_out.append((a, e))
    Wh = np.concatenate([wv[None, :], wd], 0)
    bh = np.concatenate([np.array([bv], np.float32), bd])
    out, eo = (_q8_head if q8 else _fp32_layer)(Wh, bh, a, e)
    res = dict(V=out[:, 0], head=out[:, 1:], bV=eo[:, 0], bhead=eo[:, 1:])
    raw, eraw = out[:, 1:], eo[:, 1:]
    if cfg.variant == azo.DISCRETE:
        res["post"], res["bpost"] = _softmax_bound(raw, eraw)
    else:
        K = cfg.num_components
        mu, ls = raw[:, :K], raw[:, K:2 * K]
        lsc = np.clip(ls, cfg.log_std_min, cfg.log_std_max)
        sig = np.exp(lsc)
        es = np.minimum(eraw[:, K:2 * K], 100.0)
        bsig = np.minimum(sig * np.exp(es) * (np.expm1(es) + 4 * U), np.exp(cfg.log_std_max) - np.exp(cfg.log_std_min))
        if K > 1:
            p, bp = _softmax_bound(raw[:, 2 * K:3 * K], eraw[:, 2 * K:3 * K])
        else:
            p, bp = np.ones((raw.shape[0], 1)), np.zeros((raw.shape[0], 1))
        res["post"] = np.concatenate([mu, sig, p], 1)
        res["bpost"] = np.concatenate([eraw[:, :K], bsig, bp], 1)
    if trace:
        res["layers"] = trace_out
    return res


def within(got, ref, bound):
    """Elementwise |got - ref| <= bound (NaN fails); returns (ok, worst ratio |got - ref| / bound)."""
    d = np.abs(np.asarray(got, np.float64) - ref)
    ok = bool(np.all(d <= bound))
    ratio = float(np.max(np.where(bound > 0, d / np.where(bound > 0, bound, 1), np.where(d > 0, np.inf, 0)))) if d.size else 0.0
    return ok, ratio


# ------------------------------------------------------------------------------------------------ numpy restatement of Q8


def _fmaf(a, b, c):
    """f32 fma via f64: the product of two f32 is exact in f64, the sum is rounded twice (f64, then f32).  A double rounding can
    differ from one rounding in the last bit of rare inputs, so bit equality with the oracle holds for given inputs, not in
    general (test_kernel_matrix.py checks it on its own inputs)."""
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def _act32(act, v):
    if act == azo.ACT_RELU:
        return np.where(v > 0, v, np.float32(0)).astype(np.float32)
    det_expm1f = np.vectorize(azo.lib().azo_det_expm1f, otypes=[np.float32])  # the contract's ELU (azg_oracle.c act_fn)
    return np.where(v > 0, v, det_expm1f(np.minimum(v, 0))).astype(np.float32)


def q8_contract(cfg: azo.Config, w: np.ndarray, x: np.ndarray, drop_pc=False, scale_off=None):
    """The AZO_EVAL_Q8 contract in numpy (relu / elu), layer by layer.  Returns (V, raw head, [hidden activations]).
    drop_pc: leave out the order-4 digit products PC.  scale_off = (layer, j): the scale of output j of hidden layer `layer` x 2."""
    layers, (wv, bv), (wd, bd) = split(cfg, w)
    a = np.asarray(x, np.float32).reshape(-1, cfg.state_dim)
    acts = []
    for l, (W, b) in enumerate(layers):
        if l == 0:
            y = np.broadcast_to(b, (a.shape[0], b.size)).astype(np.float32)
            for k in range(W.shape[1]):
                y = _fmaf(W[None, :, k], a[:, k:k + 1], y)
        else:
            q, uw, ew, (wh, wm, wl) = quantise_weights(W)
            vmax = np.abs(a).max(axis=1).astype(np.float32)
            ex = biased_exponent((vmax * np.float32(1.004)).astype(np.float32).astype(np.float64))
            qx = np.rint(a.astype(np.float64) / np.ldexp(1.0, ex - 149)[:, None]).astype(np.int64)
            t = (qx + 0x8080) ^ 0x8080
            xh, xm, xl = [np.where(d > 127, d - 256, d) for d in (((t >> s) & 0xFF) for s in (16, 8, 0))]
            PA, PB = xh @ wh.T, xh @ wm.T + xm @ wh.T
            PC = np.zeros_like(PA) if drop_pc else xh @ wl.T + xm @ wm.T + xl @ wh.T
            u = _fmaf(PA.astype(np.float32), np.float32(256), PB.astype(np.float32))
            u = _fmaf(u, np.float32(256), PC.astype(np.float32))
            cx = np.ldexp(1.0, ex - 149).astype(np.float32)
            cw = np.ldexp(1.0, ew - 133).astype(np.float32)
            sc = (cx[:, None] * cw[None, :]).astype(np.float32)
            if scale_off is not None and scale_off[0] == l:
                sc[:, scale_off[1]] *= np.float32(2)
            y = _fmaf(u, sc, np.broadcast_to(b, u.shape).astype(np.float32))
        a = _act32(cfg.activation, y)
        acts.append(a)
    Wh = np.concatenate([wv[None, :], wd], 0)
    bh = np.concatenate([np.array([bv], np.float32), bd])
    H = cfg.hidden
    parts = []
    for q in range(H // 32):
        s = np.zeros((a.shape[0], Wh.shape[0]), np.float32)
        for k in range(32 * q, 32 * q + 32):
            s = _fmaf(a[:, k:k + 1], Wh[None, :, k], s)
        parts.append(s)
    span = 1
    while span < len(parts):
        for q in range(0, len(parts) - span, 2 * span):
            parts[q] = (parts[q] + parts[q + span]).astype(np.float32)
        span *= 2
    out = (parts[0] + bh[None, :]).astype(np.float32)
    return out[:, 0], out[:, 1:], acts

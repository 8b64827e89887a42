"""The deterministic math, Philox and MT19937 primitives of the oracle against independent truth (CPU).

The CUDA engine (csrc/detmath.cuh, common.cuh) and the oracle (oracle/azg_oracle.c) implement these primitives op for op from
one spec, and the engine == oracle tests cannot see an error the two copies share.  These tests pin the spec itself:
  * expf / expm1f / tanhf over every f32 input of their ranges against numpy float64, with ulp bounds set at the measured
    maxima plus a hair, and their edge behaviour bit for bit;
  * sin / cos / log (f64) against x86 80-bit long double on random points, the doubles nearest k pi/2 (the hard case of the
    two-step Cody-Waite reduction), +-0, the Box-Muller grid and 1 - u of a 53-bit u;
  * the distance of each function to glibc's (DESIGN.md section 6 states it);
  * Philox4x32-10 against the known-answer vectors of Random123 (Salmon et al., SC'11);
  * the MT19937 generators of the MT19937 RNG mode against CPython's `random` and torch's CPU generator.
The GPU side (engine == oracle on the same inputs, and device-only identities) is tests/test_primitives_gpu.py.
"""
from __future__ import annotations

import ctypes
import ctypes.util
import os
import random
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from oracle import azo

THREADS = max(1, min(8, os.cpu_count() or 1))
CHUNK = 1 << 24

# (function, numpy f64 truth, f32 input range, bound in ulp of the f32 truth)
F32_CASES = {
    "expf": (np.exp, (-87.0, 88.0), 1.02),     # measured 1.010
    "expm1f": (np.expm1, (-17.5, 88.0), 1.45),  # measured 1.443
    "tanhf": (np.tanh, (-np.inf, np.inf), 1.34),  # measured 1.330 (all finite inputs)
}
# f64 functions against long double (ulp of the f64 truth) on the sets of f64_sets().  Measured maxima: sin / cos 1.063 at the
# doubles nearest k pi/2 (0x1.93c05c9ed3cbcp+19 / +18), 0.79 elsewhere; log 0.844 on 1 - u (MT mode), 0.807 on the Box-Muller grid
F64_BOUNDS = {"sin": 1.07, "cos": 1.07, "log": 0.85}

KAT = [  # Random123 kat_vectors, philox4x32_10: counter, key -> output
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
]
MT_SEEDS = [0, 1, 2**32 - 1, 2**32, 2**32 + 7, 2**63 + 5]


def kat_args(ctr, key):
    """(seed, tree, idx) of the Philox counter layout (DESIGN.md section 5) that make counter ctr and key key with stream 0,
    block 0: counter = (idx_lo, idx_hi ^ block << 16, tree_lo, tree_hi ^ stream << 24), key = (seed_lo, seed_hi)."""
    s64 = lambda lo, hi: ((hi << 32) | lo) - ((hi >> 31) << 64)  # noqa: E731  (int64 argument)
    return (key[1] << 32) | key[0], s64(ctr[2], ctr[3]), s64(ctr[0], ctr[1])


def f32_ulp_error(got: np.ndarray, truth: np.ndarray) -> np.ndarray:
    """|got - truth| in units of the f32 ulp at truth (2^-149 below the normal range)."""
    e = np.frexp(truth)[1]
    return np.abs(got.astype(np.float64) - truth) / np.ldexp(1.0, np.maximum(e - 24, -149))


def f64_ulp_error(got: np.ndarray, truth: np.ndarray) -> np.ndarray:
    """|got - truth| in units of the f64 ulp at truth (truth in long double)."""
    e = np.frexp(truth.astype(np.float64))[1]
    return np.asarray(np.abs(got.astype(np.longdouble) - truth) / np.ldexp(np.longdouble(1), np.maximum(e - 53, -1074)), np.float64)


def bit_ranges(lo: float, hi: float):
    """[start, stop) ranges of uint32 patterns covering the finite f32 values in [lo, hi] (lo < 0 < hi)."""
    pos = np.float32(min(hi, np.finfo(np.float32).max)).view(np.uint32)
    neg = np.float32(max(lo, -np.finfo(np.float32).max)).view(np.uint32)
    return [(0, int(pos) + 1), (0x80000000, int(neg) + 1)]


def chunks(ranges, size=CHUNK):
    for a, b in ranges:
        for s in range(a, b, size):
            yield s, min(b, s + size)


def _max_f32_error(fn, truth, lo, hi):
    def one(c):
        x = np.arange(c[0], c[1], dtype=np.uint32).view(np.float32)
        err = f32_ulp_error(azo.det_eval(fn, x, n_threads=1), truth(x.astype(np.float64)))
        i = int(np.argmax(err))
        return float(err[i]), float(x[i])
    with ThreadPoolExecutor(THREADS) as ex:
        return max(ex.map(one, chunks(bit_ranges(lo, hi))))


@pytest.mark.parametrize("fn", sorted(F32_CASES))
def test_f32_functions_exhaustive_ulp_bound(fn):
    """Every f32 input of the stated range: the deterministic function within its ulp bound of the f64 truth."""
    truth, (lo, hi), bound = F32_CASES[fn]
    err, at = _max_f32_error(fn, truth, lo, hi)
    assert err <= bound, f"{fn}: {err:.4f} ulp at {at!r} ({np.float32(at).view(np.uint32):#010x}), bound {bound}"


def _bits(x) -> np.ndarray:
    return np.asarray(x, np.float32).view(np.uint32)


def test_f32_function_edges():
    """The documented edge behaviour, bit for bit (signed zeros included)."""
    f32 = lambda *v: np.array(v, np.float32)  # noqa: E731
    inf, nan = np.float32(np.inf), np.float32(np.nan)
    below = np.nextafter(np.float32(-87.0), np.float32(-np.inf))
    above = np.nextafter(np.float32(88.0), np.float32(np.inf))
    assert np.array_equal(_bits(azo.det_eval("expf", f32(below, -100, -1e30, -inf))), _bits(f32(0, 0, 0, 0)))
    assert np.array_equal(_bits(azo.det_eval("expf", f32(above, 100, inf))), _bits(f32(inf, inf, inf)))
    assert np.array_equal(_bits(azo.det_eval("expf", f32(0.0, -0.0))), _bits(f32(1, 1)))
    assert np.array_equal(_bits(azo.det_eval("expm1f", f32(above, 1e30, inf))), _bits(f32(inf, inf, inf)))
    below = np.nextafter(np.float32(-17.5), np.float32(-np.inf))
    assert np.array_equal(_bits(azo.det_eval("expm1f", f32(below, -20, -1e30, -inf))), _bits(f32(-1, -1, -1, -1)))
    # expm1f(-0) is +0 (glibc: -0; harmless downstream: ELU passes it on as +0), expm1f(+0) = +0
    assert np.array_equal(_bits(azo.det_eval("expm1f", f32(-0.0, 0.0))), _bits(f32(0.0, 0.0)))
    t = f32(9.1, np.nextafter(np.float32(9.1), np.float32(20)), 100, inf)
    assert np.array_equal(_bits(azo.det_eval("tanhf", t)), _bits(f32(1, 1, 1, 1)))
    assert np.array_equal(_bits(azo.det_eval("tanhf", -t)), _bits(f32(-1, -1, -1, -1)))
    assert np.array_equal(_bits(azo.det_eval("tanhf", f32(-0.0, 0.0))), _bits(f32(-0.0, 0.0)))
    for fn in ("expf", "expm1f", "tanhf"):
        assert np.isnan(azo.det_eval(fn, f32(nan, -nan))).all(), fn


def test_activation_nan_inputs():
    """act_fn (MATH_DET) on quiet and signaling NaNs of both signs: ReLU and ReLU6 return +0 (NaN is a missing operand of the
    comparison / fmaxf, as in the engine's mlp_act), the others a NaN."""
    x = np.array([0x7F800001, 0x7FBFFFFF, 0x7FC00000, 0xFF800001, 0xFFC00001], np.uint32).view(np.float32)
    for act in (azo.ACT_RELU, azo.ACT_RELU6):
        assert np.array_equal(_bits(azo.det_eval(act, x)), np.zeros(x.size, np.uint32)), act
    for act in (azo.ACT_ELU, azo.ACT_LEAKYRELU, azo.ACT_SILU, azo.ACT_HARDSWISH):
        assert np.isnan(azo.det_eval(act, x)).all(), act


def f64_sets(n_random: int = 10_000_000):
    """The f64 inputs of the sin / cos / log accuracy tests: name -> (functions, inputs)."""
    rng = np.random.default_rng(6)
    sets = {}
    # random points |x| < 2^11: uniform mantissa, exponent spread over [2^-11, 2^11)
    x = rng.uniform(-1, 1, n_random) * np.ldexp(1.0, rng.integers(-10, 12, n_random))
    sets["random"] = (("sin", "cos"), x)
    # the doubles nearest k pi/2 (and their neighbours), k up to 2^20: |x| < 2^20 pi/2 is the stated reduction range
    k = np.arange(1, 2**20 + 1).astype(np.longdouble)
    m = (k * (np.longdouble("3.14159265358979323846264338327950288") / 2)).astype(np.float64)  # 64-bit pi: nearest but for ties
    m = np.concatenate([m, np.nextafter(m, 0), np.nextafter(m, np.inf)])
    sets["k_pi_2"] = (("sin", "cos"), np.concatenate([m, -m]))
    sets["zero"] = (("sin", "cos"), np.array([0.0, -0.0]))
    # Box-Muller grid of the noise (stream 1): u = (c + 0.5) 2^-32 and the angle 2 pi u
    c = np.concatenate([rng.integers(0, 2**32, n_random // 4, dtype=np.uint64), np.arange(4096, dtype=np.uint64),
                        2**32 - 1 - np.arange(4096, dtype=np.uint64)])
    u = (c.astype(np.float64) + 0.5) * 2.3283064365386963e-10
    sets["bm_log"] = (("log",), u)
    sets["bm_angle"] = (("sin", "cos"), 6.283185307179586 * u)
    # MT mode: -log1p(-u) = -log(1 - u) with a 53-bit uniform u (1 - u exact)
    u53 = rng.integers(0, 2**53, n_random // 4, dtype=np.uint64).astype(np.float64) * 2.0**-53
    u53 = np.concatenate([u53, np.arange(4096) * 2.0**-53, 1 - np.arange(1, 4096) * 2.0**-53])
    sets["mt_log"] = (("log",), 1.0 - u53)
    return sets


_LD = {"sin": np.sin, "cos": np.cos, "log": np.log}


def _libm():
    return ctypes.CDLL(ctypes.util.find_library("m"))


def test_f64_functions_against_long_double():
    """sin / cos / log within their bounds of the long double truth on every set; sin(+-0) = +0 and cos(+-0) = 1 exactly."""
    worst = {}
    for name, (fns, x) in f64_sets().items():
        for fn in fns:
            got = azo.det_eval(fn, x, n_threads=THREADS)
            parts = np.array_split(np.arange(x.size), THREADS)
            with ThreadPoolExecutor(THREADS) as ex:
                errs = list(ex.map(lambda ix: f64_ulp_error(got[ix], _LD[fn](x[ix].astype(np.longdouble))), parts))
            err = np.concatenate(errs)
            i = int(np.argmax(err))
            worst[(name, fn)] = (float(err[i]), float(x[i]).hex())
            assert err[i] <= F64_BOUNDS[fn], f"{fn} on {name}: {err[i]:.4f} ulp at {float(x[i]).hex()}"
    z = np.array([0.0, -0.0])
    assert np.array_equal(azo.det_eval("sin", z).view(np.uint64), np.zeros(2, np.uint64))  # +0 for both (glibc: sin(-0) = -0)
    assert np.array_equal(azo.det_eval("cos", z), np.ones(2))
    assert azo.det_eval("log", np.array([1.0]))[0] == 0.0


def _ordered(a: np.ndarray) -> np.ndarray:
    """Map floats to integers whose differences count representable values between them."""
    it = np.int64 if a.dtype == np.float64 else np.int32
    i = a.view(it).astype(np.int64)
    return np.where(i < 0, np.int64(np.iinfo(it).min) - i, i)


def test_distance_to_glibc():
    """DESIGN.md section 6: distance to glibc in representable values: expf 1, expm1f 2, tanhf 2 (the worst inputs over all f32,
    measured exhaustively, are listed), sin / cos / log 1 (on a sample of the f64 sets)."""
    libm = _libm()
    for n in ("expf", "expm1f", "tanhf"):
        getattr(libm, n).restype, getattr(libm, n).argtypes = ctypes.c_float, [ctypes.c_float]
    for n in ("sin", "cos", "log"):
        getattr(libm, n).restype, getattr(libm, n).argtypes = ctypes.c_double, [ctypes.c_double]
    rng = np.random.default_rng(7)
    known = {"expf": float.fromhex("0x1p-24"), "expm1f": float.fromhex("0x1.63008ap-2"), "tanhf": float.fromhex("0x1.f72258p-7")}
    limit = {"expf": 1, "expm1f": 2, "tanhf": 2}
    for fn, (_, (lo, hi), _) in F32_CASES.items():
        x = np.concatenate([rng.uniform(max(lo, -40.0), min(hi, 40.0), 20000), [known[fn]]]).astype(np.float32)
        got = azo.det_eval(fn, x)
        ref = np.array([getattr(libm, fn)(float(v)) for v in x], np.float32)
        d = np.abs(_ordered(got) - _ordered(ref))
        assert d.max() <= limit[fn], fn
        assert d[-1] == limit[fn], f"{fn} at {float(x[-1]).hex()}: {d[-1]}"
    for name, (fns, x) in f64_sets(200_000).items():
        x = x[rng.permutation(x.size)[:5000]]
        for fn in fns:
            got = azo.det_eval(fn, x)
            ref = np.array([getattr(libm, fn)(float(v)) for v in x])
            assert np.abs(_ordered(got) - _ordered(ref)).max() <= 1, (name, fn)


@pytest.mark.parametrize("ctr,key,out", KAT)
def test_philox_known_answers(ctr, key, out):
    seed, tree, idx = kat_args(ctr, key)
    assert tuple(azo.rng_u32(seed, tree, 0, idx, 0, w) for w in range(4)) == out


@pytest.mark.parametrize("seed", MT_SEEDS)
def test_mt19937_python_mode_equals_cpython(seed):
    """random.seed(seed) (init_by_array; two key words from 2^32 on), random() past the 624-output regeneration, _randbelow(n)
    for n = 1..40 with equal draw counts (the next getrandbits(32) agrees), then raw outputs."""
    ref = random.Random(seed)
    g = azo.MT19937(seed, "python")
    for _ in range(400):
        assert g.random() == ref.random()
    for n in range(1, 41):
        for _ in range(5):
            assert g.below(n) == ref.randrange(n)
        assert g.u32() == ref.getrandbits(32)
    for _ in range(700):
        assert g.u32() == ref.getrandbits(32)


@pytest.mark.parametrize("seed", MT_SEEDS)
def test_mt19937_torch_mode_equals_torch(seed):
    """torch.manual_seed(seed) then one-element float64 torch.rand calls (torch's scalar path: 53 bits of two outputs)."""
    torch = pytest.importorskip("torch")
    ref = torch.Generator().manual_seed(seed)
    g = azo.MT19937(seed, "torch")
    for _ in range(700):  # 1400 outputs: two regenerations
        assert g.uniform() == torch.rand(1, dtype=torch.float64, generator=ref).item()

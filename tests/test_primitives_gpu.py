"""The engine's numeric and random primitives on the device: device == oracle bit for bit, and device-only identities.

tests/primitives_probe.cu wraps each primitive of the engine headers (detmath.cuh, mlp.cuh, common.cuh, tree_discrete.cuh) in an
elementwise kernel; the module fixture compiles it with the engine's nvcc flags into a temporary directory.  The tests here:
  * expf_ / expm1f_ / tanhf_ and mlp_act<ACT> for all six activations on every one of the 2^32 f32 bit patterns, equal to the
    oracle bit for bit (signed zeros included; NaN only has to map to NaN), and the three functions within the ulp bounds of
    tests/test_primitives.py against an f64 evaluation on the device;
  * mlp_act2<ACT> (f32x2 packed) == mlp_act<ACT> per lane, exhaustively, with a different permutation of the patterns in .y;
  * sin_ / cos_ / sincos_ / log_ == oracle on the sets of the CPU test and on the whole Box-Muller grid (all 2^32 c);
  * the reciprocal-table division (div_small, div_tab + div_tab_ok, sqrt_small) == IEEE division / sqrt, and ds_decide == a
    numpy restatement with plain division;
  * the three Philox copies against the Random123 known answers and the oracle, u32_to_unit / u32_to_index against their
    integer formulas, the MT19937 copies against CPython and torch;
  * env edges through azg_env_step against the oracle and a plain-Python restatement of gym.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import random
import shutil
import subprocess

import numpy as np
import pytest

from oracle import azo
from test_primitives import F32_CASES, KAT, MT_SEEDS, bit_ranges, chunks, f64_sets, kat_args

pytestmark = pytest.mark.gpu

PROBE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "primitives_probe.cu")
CH = 1 << 26                      # elements per chunk of an exhaustive sweep
ALL = [(0, 1 << 32)]
F32_FN = {"expf": 0, "expm1f": 1, "tanhf": 2}
ACTS = [azo.ACT_RELU, azo.ACT_ELU, azo.ACT_LEAKYRELU, azo.ACT_RELU6, azo.ACT_SILU, azo.ACT_HARDSWISH]
PERM_MUL, PERM_ADD = 0x9E3779B1, 0x7F4A7C15  # lane .y of the mlp_act2 sweep: bits = PERM_MUL * i + PERM_ADD (a permutation)
AZG_TAB, FUSED_TAB = 1024, 255
THREADS = os.cpu_count() or 1  # oracle threads of the exhaustive comparisons

vp, i32, u32, i64, u64, f64 = C.c_void_p, C.c_int32, C.c_uint32, C.c_int64, C.c_uint64, C.c_double
SIGS = {
    "probe_f32": [i32, vp, u32, u32, u64, vp, i64, vp],
    "probe_f32_truth": [i32, vp, u32, u32, u64, vp, i64, vp],
    "probe_act2": [i32, u32, u32, u32, u32, u64, vp, vp, i64, vp],
    "probe_f64": [i32, vp, u64, vp, vp, i64, vp],
    "probe_div": [i32, vp, vp, vp, vp, i32, vp, i64, vp],
    "probe_ds_decide": [vp, vp, vp, vp, vp, i32, f64, i32, vp, i64, vp],
    "probe_philox": [i32, u64, vp, vp, vp, vp, i32, vp, i64, vp],
    "probe_u32_map": [vp, vp, vp, vp, i64, vp],
    "probe_mt": [i32, vp, i32, vp, i32, vp, vp],
}


class Probe:
    def __init__(self, path):
        import torch
        self.torch = torch
        self.L = C.CDLL(path)
        for name, args in SIGS.items():
            f = getattr(self.L, name)
            f.restype, f.argtypes = C.c_int, args

    def __call__(self, name, *args):
        conv = [a.data_ptr() if isinstance(a, self.torch.Tensor) else a for a in args]
        rc = getattr(self.L, name)(*conv, self.torch.cuda.current_stream().cuda_stream)
        assert rc == 0, f"{name}: CUDA error {rc}"


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    import torch
    from alphazero_gym_b200.build import NVCC_FLAGS
    assert torch.cuda.is_available()
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    out = str(tmp_path_factory.mktemp("probe") / "primitives_probe.so")
    res = subprocess.run([nvcc, *NVCC_FLAGS, "-o", out, PROBE], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    return Probe(out)


def _t():
    import torch
    return torch


def u32_of(x):
    """uint32 bit patterns of a float32 tensor / array, as int64 (torch) or uint32 (numpy)."""
    if isinstance(x, np.ndarray):
        return x.view(np.uint32)
    return x.view(_t().int32).to(_t().int64) & 0xFFFFFFFF


def assert_f32_equal(got, ref, what):
    """Bitwise equality of float32 arrays; a NaN only has to meet a NaN."""
    if np.array_equal(got.view(np.uint32), ref.view(np.uint32)):
        return
    bad = (got.view(np.uint32) != ref.view(np.uint32)) & ~(np.isnan(got) & np.isnan(ref))
    if bad.any():
        i = np.flatnonzero(bad)
        raise AssertionError(f"{what}: {i.size} patterns differ, e.g. input #{i[0]}: {got[i[0]]!r} vs {ref[i[0]]!r}")


def assert_f32_equal_dev(got, ref, what):
    torch = _t()
    bad = (u32_of(got) != u32_of(ref)) & ~(torch.isnan(got) & torch.isnan(ref))
    n = int(bad.sum())
    assert n == 0, f"{what}: {n} patterns differ, e.g. {int(torch.nonzero(bad)[0])}"


# ---- f32 functions and activations, exhaustive ------------------------------------------------------------------------------------
@pytest.mark.parametrize("fn", list(F32_FN) + [f"act{a}" for a in ACTS])
def test_f32_device_equals_oracle_exhaustive(probe, fn):
    """Every f32 bit pattern: det::expf_ / expm1f_ / tanhf_ and mlp_act<ACT> == the oracle's functions / act_fn (MATH_DET)."""
    torch = _t()
    code, ofn = (F32_FN[fn], fn) if fn in F32_FN else (16 + int(fn[3:]), int(fn[3:]))
    out = torch.empty(CH, dtype=torch.float32, device="cuda")
    host = torch.empty(CH, dtype=torch.float32, pin_memory=True)
    idx = np.arange(CH, dtype=np.uint32)
    for s, e in chunks(ALL, CH):
        probe("probe_f32", code, None, 1, 0, s, out, e - s)
        host.copy_(out)
        x = (idx + np.uint32(s)).view(np.float32)
        assert_f32_equal(host.numpy(), azo.det_eval(ofn, x, n_threads=THREADS), f"{fn} chunk {s:#x}")


@pytest.mark.parametrize("fn", sorted(F32_CASES))
def test_f32_device_accuracy_exhaustive(probe, fn):
    """The CPU test's ulp bounds, checked on the device against libdevice exp / expm1 / tanh in double."""
    torch = _t()
    _, (lo, hi), bound = F32_CASES[fn]
    got = torch.empty(CH, dtype=torch.float32, device="cuda")
    tru = torch.empty(CH, dtype=torch.float64, device="cuda")
    worst = 0.0
    for s, e in chunks(bit_ranges(lo, hi), CH):
        probe("probe_f32", F32_FN[fn], None, 1, 0, s, got, e - s)
        probe("probe_f32_truth", F32_FN[fn], None, 1, 0, s, tru, e - s)
        g, t = got[:e - s].double(), tru[:e - s]
        ex = torch.frexp(t).exponent.to(torch.int64)
        ulp = torch.pow(2.0, torch.clamp(ex - 24, min=-149).double())
        worst = max(worst, float(((g - t).abs() / ulp).max()))
    assert worst <= bound, f"{fn}: {worst:.4f} ulp, bound {bound}"


@pytest.mark.parametrize("act", ACTS)
def test_mlp_act2_equals_mlp_act_exhaustive(probe, act):
    """mlp_act2<ACT> (f32x2) == mlp_act<ACT> per lane: .x over every pattern in order, .y over a different permutation."""
    torch = _t()
    ox, oy, rx, ry = (torch.empty(CH, dtype=torch.float32, device="cuda") for _ in range(4))
    for s, e in chunks(ALL, CH):
        n = e - s
        probe("probe_act2", act, 1, 0, PERM_MUL, PERM_ADD, s, ox, oy, n)
        probe("probe_f32", 16 + act, None, 1, 0, s, rx, n)
        probe("probe_f32", 16 + act, None, PERM_MUL, PERM_ADD, s, ry, n)
        assert_f32_equal_dev(ox[:n], rx[:n], f"act {act} lane x chunk {s:#x}")
        assert_f32_equal_dev(oy[:n], ry[:n], f"act {act} lane y chunk {s:#x}")


# ---- f64 sin / cos / log ----------------------------------------------------------------------------------------------------------
def _f64_dev(probe, fn, x):
    torch = _t()
    xd = torch.from_numpy(np.ascontiguousarray(x, np.float64)).cuda()
    a, b = torch.empty_like(xd), torch.empty_like(xd)
    probe("probe_f64", fn, xd, 0, a, b, xd.numel())
    return a.cpu().numpy(), b.cpu().numpy()


def test_f64_device_equals_oracle_on_sets(probe):
    """sin_, cos_, sincos_ and log_ == oracle bit for bit on the CPU test's sets (random, k pi/2, +-0, Box-Muller, 1 - u)."""
    for name, (fns, x) in f64_sets().items():
        if "log" in fns:
            got, _ = _f64_dev(probe, 3, x)
            assert np.array_equal(got.view(np.uint64), azo.det_eval("log", x, THREADS).view(np.uint64)), name
            continue
        rs, rc = azo.det_eval("sin", x, THREADS).view(np.uint64), azo.det_eval("cos", x, THREADS).view(np.uint64)
        s, _ = _f64_dev(probe, 0, x)
        c, _ = _f64_dev(probe, 1, x)
        ss, cc = _f64_dev(probe, 2, x)
        for got, ref, what in ((s, rs, "sin_"), (c, rc, "cos_"), (ss, rs, "sincos_ s"), (cc, rc, "sincos_ c")):
            assert np.array_equal(got.view(np.uint64), ref), f"{what} on {name}"


def test_f64_device_equals_oracle_box_muller_grid_exhaustive(probe):
    """log_(u) and sincos_(2 pi u) for every u = (c + 0.5) 2^-32 of the noise's Box-Muller transform == oracle."""
    torch = _t()
    lg, s, c = (torch.empty(CH, dtype=torch.float64, device="cuda") for _ in range(3))
    idx = np.arange(CH, dtype=np.float64)
    for b, e in chunks(ALL, CH):
        probe("probe_f64", 4, None, b, lg, lg, e - b)
        probe("probe_f64", 5, None, b, s, c, e - b)
        u = (idx + float(b) + 0.5) * 2.3283064365386963e-10
        ang = 6.283185307179586 * u
        for dev, ref, what in ((lg, azo.det_eval("log", u, THREADS), "log"), (s, azo.det_eval("sin", ang, THREADS), "sin"),
                               (c, azo.det_eval("cos", ang, THREADS), "cos")):
            assert np.array_equal(dev.cpu().numpy().view(np.uint64), ref.view(np.uint64)), f"{what} chunk {b:#x}"


# ---- reciprocal-table division ----------------------------------------------------------------------------------------------------
def engine_tables():
    """rcp[i] = 1 / i and sq[i] = sqrt(i) for i <= AZG_TAB, built as azg_create builds them (IEEE division and sqrt)."""
    i = np.arange(AZG_TAB + 1, dtype=np.float64)
    with np.errstate(divide="ignore"):
        rcp = np.where(i > 0, 1.0 / np.maximum(i, 1), 0.0)
    return rcp, np.sqrt(i)


def div_tab_ok_np(a: np.ndarray) -> np.ndarray:
    e = (a.view(np.uint64) >> np.uint64(52)) & np.uint64(0x7FF)
    return (e >= 0xC2) & (e < 0xC2 + 0x67B)


def numerators(rng) -> np.ndarray:
    """The numerators of the division tests (see test_table_division_equals_ieee)."""
    ints = np.arange(-2000, 2001, dtype=np.float64)
    parts = [
        rng.integers(0, 0x7FF0 << 48, 4000, dtype=np.uint64).view(np.float64) * rng.choice([-1.0, 1.0], 4000),  # whole exponent range
        ints, ints + 0.5, ints * 37.25, rng.integers(-10**6, 10**6, 2000).astype(np.float64),                      # CartPole W sums
    ]
    sq = np.sqrt(np.arange(1, 1101, dtype=np.float64))                                                          # values near sqrt(i)
    parts += [sq, np.nextafter(sq, 0), np.nextafter(sq, np.inf), np.nextafter(np.nextafter(sq, 0), 0)]
    e = np.array([0xC1, 0xC2, 0xC3, 0xC2 + 0x679, 0xC2 + 0x67A, 0xC2 + 0x67B, 0xC2 + 0x67C], np.uint64)      # div_tab_ok window edges
    mant = rng.integers(0, 1 << 52, (e.size, 40), dtype=np.uint64)
    mant[:, 0], mant[:, 1] = 0, (1 << 52) - 1
    edge = ((e[:, None] << np.uint64(52)) | mant).ravel().view(np.float64)
    parts += [edge, -edge]
    g = np.array([1e-250, 1e250])                                                                                 # div_small's guard
    g = np.concatenate([g, np.nextafter(g, 0), np.nextafter(g, np.inf)])
    parts += [g, -g]
    parts.append(np.array([0.0, -0.0, 5e-324, -5e-324, 2.2250738585072014e-308, 1e-310, np.inf, -np.inf, np.nan]))
    return np.concatenate(parts)


def near_midpoints(rng, b: np.ndarray) -> np.ndarray:
    """For each divisor b, numerators a = RN(b (m + ulp(m) / 2)) with random m: quotients next to a rounding midpoint, the hard case
    of a one-step correction (an exact midpoint quotient of a double by an integer does not exist), and their neighbours."""
    m = 1.0 + rng.integers(0, 1 << 52, (b.size, 8), dtype=np.uint64).astype(np.float64) * 2.0**-52
    m = m * np.ldexp(1.0, rng.integers(-30, 30, m.shape))
    half = np.ldexp(1.0, np.frexp(m)[1] - 54).astype(np.longdouble)
    a = (b[:, None].astype(np.longdouble) * (m.astype(np.longdouble) + half)).astype(np.float64)
    return np.stack([a, np.nextafter(a, 0), np.nextafter(a, np.inf)], -1).reshape(b.size, -1)


def _div_dev(probe, which, a, b, rcp, sq, tabn):
    torch = _t()
    ad = torch.from_numpy(np.ascontiguousarray(a, np.float64)).cuda()
    bd = torch.from_numpy(np.ascontiguousarray(b, np.int32)).cuda()
    out = torch.empty_like(ad)
    probe("probe_div", which, ad, bd, rcp, sq, tabn, out, ad.numel())
    return out.cpu().numpy()


def _same(x, y):
    """Bitwise equality of float64 arrays (signed zeros included); a NaN only has to meet a NaN."""
    return bool(np.all((x.view(np.uint64) == y.view(np.uint64)) | (np.isnan(x) & np.isnan(y))))


def test_table_division_equals_ieee(probe):
    """div_small(a, b) (tables of 1024 and 255 entries) and div_tab(a, b) wherever div_tab_ok(a) == __ddiv_rn(a, b) == numpy a / b,
    for every b in 1..1100 and numerators: random over the exponent range, integers and half-integers, values near sqrt(i),
    near-midpoint quotients, the div_tab_ok window edges, the 1e-250 / 1e250 guard, +-0, subnormals, +-inf, NaN.  sqrt_small(n) ==
    sqrt(n) up to 1100; div_tab_ok == its definition."""
    torch = _t()
    rng = np.random.default_rng(11)
    rcp_h, sq_h = engine_tables()
    rcp, sq = torch.from_numpy(rcp_h).cuda(), torch.from_numpy(sq_h).cuda()
    b = np.arange(1, 1101, dtype=np.int32)
    num = numerators(rng)
    A = np.concatenate([np.broadcast_to(num, (b.size, num.size)), near_midpoints(rng, b.astype(np.float64))], 1)
    B = np.broadcast_to(b[:, None], A.shape)
    A, B = A.ravel(), np.ascontiguousarray(B).ravel()
    with np.errstate(all="ignore"):
        ref = A / B
    assert _same(_div_dev(probe, 2, A, B, rcp, sq, AZG_TAB), ref), "__ddiv_rn differs from numpy"
    for tabn in (AZG_TAB, FUSED_TAB):
        got = _div_dev(probe, 0, A, B, rcp, sq, tabn)
        bad = ~((got.view(np.uint64) == ref.view(np.uint64)) | (np.isnan(got) & np.isnan(ref)))
        assert not bad.any(), f"div_small (tabn {tabn}): {bad.sum()} cases, e.g. {A[bad][0]!r} / {B[bad][0]}"
    ok = _div_dev(probe, 3, A, B, rcp, sq, AZG_TAB) == 1.0
    assert np.array_equal(ok, div_tab_ok_np(A))
    m = ok & (B <= AZG_TAB)
    got = _div_dev(probe, 1, A[m], B[m], rcp, sq, AZG_TAB)
    assert np.array_equal(got.view(np.uint64), ref[m].view(np.uint64)), "div_tab differs from a / b inside its window"
    n = np.arange(0, 1101, dtype=np.int32)
    for tabn in (AZG_TAB, FUSED_TAB):
        got = _div_dev(probe, 4, np.zeros(n.size), n, rcp, sq, tabn)
        assert np.array_equal(got, np.sqrt(n.astype(np.float64))), f"sqrt_small (tabn {tabn})"


# ---- ds_decide ----------------------------------------------------------------------------------------------------------------------
def ds_decide_np(W, cnt, f, c_uct, puct_f32):
    """mcts.py:483-484 + helpers.argmax with plain division and sqrt: bit 0 = argmax, bit 1 = tie, bit 2 = NaN."""
    n0, n1, nn = cnt[:, 0].astype(np.float64), cnt[:, 1].astype(np.float64), cnt[:, 2].astype(np.float64)
    pr = f[:, :2]
    V = f[:, 2].astype(np.float64)
    if puct_f32:
        pc = (pr * np.float32(c_uct)).astype(np.float64)
    else:
        pc = pr.astype(np.float64) * c_uct
    sq = np.sqrt(nn)
    with np.errstate(all="ignore"):
        u0 = np.where(n0 > 0, W[:, 0] / n0, V) + pc[:, 0] * (sq / (n0 + 1))
        u1 = np.where(n1 > 0, W[:, 1] / n1, V) + pc[:, 1] * (sq / (n1 + 1))
    return ((u1 > u0).astype(np.uint32) | ((u0 == u1).astype(np.uint32) << 1)
            | ((np.isnan(u0) | np.isnan(u1)).astype(np.uint32) << 2))


def ds_cases(rng, n=200_000):
    nn = rng.integers(1, 600, n)
    n0 = (rng.random(n) * nn).astype(np.int64)
    n1 = (rng.random(n) * nn).astype(np.int64)
    k = rng.integers(0, 6, n)
    n0 = np.where(k == 0, nn - 1, n0)                          # n == nn - 1
    n1 = np.where(k == 1, nn - 1, n1)
    n0 = np.where(k == 2, nn + rng.integers(0, 3, n), n0)      # n >= nn: the checked path
    W = np.stack([np.where(rng.random(n) < 0.5, rng.integers(0, 2, n) * n0 * rng.random(n), rng.integers(-5, 200, n) * 1.0),
                  np.where(rng.random(n) < 0.5, rng.normal(0, 50, n), rng.integers(0, 200, n) * 1.0)], 1)
    f = np.stack([rng.random(n), rng.random(n), rng.normal(0, 20, n)], 1).astype(np.float32)
    # exact ties: equal statistics on both edges; equal W / n with equal priors and counts; unvisited edges with equal priors
    t = rng.random(n) < 0.2
    n1 = np.where(t, n0, n1)
    W[t, 1] = W[t, 0]
    f[t, 1] = f[t, 0]
    z = rng.random(n) < 0.05
    n0[z], n1[z] = 0, 0
    f[z, 1] = f[z, 0]
    # NaN W or V
    W[rng.random(n) < 0.01, 0] = np.nan
    f[rng.random(n) < 0.01, 2] = np.nan
    cnt = np.stack([n0, n1, nn], 1).astype(np.int32)
    return np.ascontiguousarray(W), np.ascontiguousarray(cnt), np.ascontiguousarray(f)


@pytest.mark.parametrize("puct_f32", [1, 0])
@pytest.mark.parametrize("c_uct", [1.5, 0.05])
def test_ds_decide_equals_plain_division(probe, puct_f32, c_uct):
    """The cached selection rule of the shared-memory CartPole kernel (255-entry tables) == a numpy restatement with plain / and
    sqrt, on random statistics (n == nn - 1, nn > 255 and n >= nn included), exact ties and NaN W or V."""
    torch = _t()
    rcp_h, sq_h = engine_tables()
    rcp, sq = torch.from_numpy(rcp_h).cuda(), torch.from_numpy(sq_h).cuda()
    W, cnt, f = ds_cases(np.random.default_rng(12 + puct_f32))
    out = torch.empty(W.shape[0], dtype=torch.int32, device="cuda")
    probe("probe_ds_decide", torch.from_numpy(W).cuda(), torch.from_numpy(cnt).cuda(), torch.from_numpy(f).cuda(), rcp, sq, FUSED_TAB,
          c_uct, puct_f32, out, W.shape[0])
    got = out.cpu().numpy().view(np.uint32)
    ref = ds_decide_np(W, cnt, f, c_uct, puct_f32)
    bad = np.flatnonzero(got != ref)
    assert bad.size == 0, f"{bad.size} cases differ, e.g. W={W[bad[0]]} cnt={cnt[bad[0]]} f={f[bad[0]]}: {got[bad[0]]} vs {ref[bad[0]]}"
    assert (ref & 2).sum() > 1000 and (ref & 4).sum() > 100 and ((ref & 6) == 0).sum() > 10000  # the cases reach all outcomes


# ---- Philox -------------------------------------------------------------------------------------------------------------------------
def _philox_dev(probe, which, seed, tree, stream, idx, block, stride=2):
    torch = _t()
    n = len(tree)
    cv = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).cuda()  # noqa: E731
    out = torch.empty((n, 4) if which < 2 else n, dtype=torch.int32, device="cuda")
    probe("probe_philox", which, seed, cv(tree, np.int64), cv(stream, np.int32), cv(idx, np.int64), cv(block, np.int32), stride, out, n)
    return out.cpu().numpy().view(np.uint32)


def test_philox_known_answers_on_device(probe):
    """rng_block reproduces all three Random123 vectors; philox_draw_x and rng_select_u32x4 (stream 0, block 0 only) vector 1."""
    for ctr, key, out in KAT:
        seed, tree, idx = kat_args(ctr, key)
        assert tuple(_philox_dev(probe, 0, seed, [tree], [0], [idx], [0])[0]) == out
    seed, tree, idx = kat_args(*KAT[0][:2])
    assert _philox_dev(probe, 2, seed, [tree], [0], [idx], [0])[0] == KAT[0][2][0]
    assert _philox_dev(probe, 1, seed, [tree], [0], [idx], [0], stride=1)[0][0] == KAT[0][2][0]


def test_philox_copies_equal_oracle(probe):
    """rng_block, rng_select_u32x4 and philox_draw_x == the oracle on 2^24 random counters: tree ids >= 2^32, streams 0-3, blocks up
    to 2^15, draw indices up to 2^31 - 1."""
    rng = np.random.default_rng(13)
    n = 1 << 24
    seed = int(rng.integers(0, 2**63)) * 2 + 1
    tree = rng.integers(2**32, 2**62, n)
    tree[:1000] = rng.integers(0, 2**32, 1000)
    stream = rng.integers(0, 4, n)
    block = rng.integers(0, 2**15, n)
    idx = rng.integers(0, 2**31 - 7, n)
    idx[:4] = [0, 1, 2**31 - 8, 2**31 - 7]
    ref = azo.rng_blocks(seed, tree, stream, idx, block)
    assert np.array_equal(_philox_dev(probe, 0, seed, tree, stream, idx, block), ref), "rng_block"
    zero = np.zeros(n, np.int32)
    ref0 = azo.rng_blocks(seed, tree, zero, idx, zero)[:, 0]
    assert np.array_equal(_philox_dev(probe, 2, seed, tree, zero, idx, zero), ref0), "philox_draw_x"
    m = n // 4
    x4 = _philox_dev(probe, 1, seed, tree[:m], zero[:m], idx[:m], zero[:m], stride=2)
    for q in range(4):
        refq = azo.rng_blocks(seed, tree[:m], zero[:m], idx[:m] + 2 * q, zero[:m])[:, 0]
        assert np.array_equal(x4[:, q], refq), f"rng_select_u32x4 draw {q}"


def test_u32_to_unit_and_index(probe):
    """u32_to_unit(x) = (x >> 8) 2^-24 and u32_to_index(x, n) = (x n) >> 32: every x for n = 2, random x for n = 1..16."""
    torch = _t()
    unit = torch.empty(CH, dtype=torch.float32, device="cuda")
    index = torch.empty(CH, dtype=torch.int32, device="cuda")
    two = torch.full((CH,), 2, dtype=torch.int32, device="cuda")
    for s, e in chunks(ALL, CH):
        x = torch.arange(s, e, dtype=torch.int64, device="cuda")
        probe("probe_u32_map", torch.where(x >= 2**31, x - 2**32, x).to(torch.int32), two, unit, index, e - s)
        assert torch.equal(unit[:e - s].double(), (x >> 8).double() * 2.0**-24), f"u32_to_unit chunk {s:#x}"
        assert torch.equal(index[:e - s].long(), (x * 2) >> 32), f"u32_to_index(x, 2) chunk {s:#x}"
    rng = np.random.default_rng(14)
    x = rng.integers(0, 2**32, 1 << 22, dtype=np.uint64)
    m = rng.integers(1, 17, x.size)
    xd = torch.from_numpy(x.astype(np.uint32).view(np.int32)).cuda()
    md = torch.from_numpy(m.astype(np.int32)).cuda()
    u, ix = torch.empty(x.size, dtype=torch.float32, device="cuda"), torch.empty(x.size, dtype=torch.int32, device="cuda")
    probe("probe_u32_map", xd, md, u, ix, x.size)
    assert np.array_equal(ix.cpu().numpy(), ((x * m.astype(np.uint64)) >> np.uint64(32)).astype(np.int32))
    assert np.array_equal(u.cpu().numpy().astype(np.float64), (x >> np.uint64(8)).astype(np.float64) * 2.0**-24)


# ---- MT19937 ------------------------------------------------------------------------------------------------------------------------
def mt_ops():
    """400 random(), then for n = 1..40 five _randbelow(n) and one raw output, then 700 raw outputs (past two regenerations)."""
    ops = [-1] * 400
    for n in range(1, 41):
        ops += [n] * 5 + [0]
    return np.array(ops + [0] * 700, np.int32)


def test_mt19937_device_equals_cpython_and_torch(probe):
    torch = _t()
    seeds = torch.from_numpy(np.array(MT_SEEDS, np.uint64).view(np.int64)).cuda()
    ops = mt_ops()
    out = torch.empty((len(MT_SEEDS), ops.size), dtype=torch.float64, device="cuda")
    probe("probe_mt", 0, seeds, len(MT_SEEDS), torch.from_numpy(ops).cuda(), ops.size, out)
    got = out.cpu().numpy()
    for t, s in enumerate(MT_SEEDS):
        ref = random.Random(s)
        exp = [ref.random() if o < 0 else (ref.getrandbits(32) if o == 0 else ref.randrange(o)) for o in ops]
        assert np.array_equal(got[t], np.array(exp, np.float64)), f"CPython seed {s}"
    nt = 700
    out = torch.empty((len(MT_SEEDS), nt), dtype=torch.float64, device="cuda")
    probe("probe_mt", 1, seeds, len(MT_SEEDS), torch.zeros(nt, dtype=torch.int32, device="cuda"), nt, out)
    got = out.cpu().numpy()
    for t, s in enumerate(MT_SEEDS):
        g = torch.Generator().manual_seed(s)
        exp = [torch.rand(1, dtype=torch.float64, generator=g).item() for _ in range(nt)]
        assert np.array_equal(got[t], np.array(exp)), f"torch seed {s}"


# ---- env edges ----------------------------------------------------------------------------------------------------------------------
def gym_pendulum(th, thdot, u):
    """gym Pendulum-v0 step with math.sin and Python's float modulo (the action clipped as an f32, then promoted)."""
    g, m, l, dt = 10.0, 1.0, 1.0, 0.05
    u = float(np.clip(np.float32(u), np.float32(-2.0), np.float32(2.0)))
    an = ((th + math.pi) % (2 * math.pi)) - math.pi
    costs = an * an + 0.1 * (thdot * thdot) + 0.001 * (u * u)
    newthdot = thdot + (-3 * g / (2 * l) * math.sin(th + math.pi) + 3.0 / (m * l * l) * u) * dt
    newth = th + newthdot * dt
    newthdot = min(max(newthdot, -8.0), 8.0) if newthdot == newthdot else newthdot
    return (newth, newthdot), -costs, False


def gym_cartpole(s, action):
    x, x_dot, theta, theta_dot = s
    gravity, masscart, masspole, length, force_mag, tau = 9.8, 1.0, 0.1, 0.5, 10.0, 0.02
    total_mass, polemass_length = masspole + masscart, masspole * length
    force = force_mag if action == 1 else -force_mag
    costheta, sintheta = math.cos(theta), math.sin(theta)
    temp = (force + polemass_length * theta_dot * theta_dot * sintheta) / total_mass
    thetaacc = (gravity * sintheta - costheta * temp) / (length * (4.0 / 3.0 - masspole * costheta * costheta / total_mass))
    xacc = temp - polemass_length * thetaacc * costheta / total_mass
    x, x_dot = x + tau * x_dot, x_dot + tau * xacc
    theta, theta_dot = theta + tau * theta_dot, theta_dot + tau * thetaacc
    thr = 12 * 2 * math.pi / 360
    return (x, x_dot, theta, theta_dot), 1.0, x < -2.4 or x > 2.4 or theta < -thr or theta > thr


def pendulum_edge_cases():
    pi = math.pi
    wrap = [th for th in (k * (2 * pi) - pi for k in range(-60, 61)) if math.fmod(th + pi, 2 * pi) == 0.0]
    assert len(wrap) > 10
    rng = np.random.default_rng(15)
    ths = wrap + [-pi, 0.0, -0.0, -1e5, 1e5, -12345.678] + list(rng.uniform(-1e5, 1e5, 40)) + list(-rng.uniform(0, 50, 40))
    two = np.float32(2.0)
    acts = [2.0, -2.0, float(np.nextafter(two, np.float32(3))), float(np.nextafter(two, np.float32(0))),
            -float(np.nextafter(two, np.float32(3))), -float(np.nextafter(two, np.float32(0))), 0.0, 0.7, float("nan")]
    cases = [(th, td, a) for th in ths for td in (0.0, -3.0, 7.9) for a in acts]
    # thdot landing on +-8: sin(th + pi) = 0 at th = -pi, so newthdot = thdot + 3 u dt
    cases += [(-pi, td, a) for td in (8.0, -8.0, 7.7, -7.7, 7.85, -7.85, float(np.nextafter(8.0, 9)), float(np.nextafter(-8.0, -9)))
              for a in (0.0, 1.0, -1.0, 2.0, -2.0)]
    return cases


def cartpole_edge_cases():
    thr = 12 * 2 * math.pi / 360
    xs = [2.4, -2.4, math.nextafter(2.4, 3), math.nextafter(2.4, 0), math.nextafter(-2.4, -3), math.nextafter(-2.4, 0)]
    ths = [thr, -thr, math.nextafter(thr, 1), math.nextafter(thr, 0), math.nextafter(-thr, -1), math.nextafter(-thr, 0)]
    cases = [((x, 0.0, 0.0, 0.0), a) for x in xs for a in (0, 1)]
    cases += [((0.0, 0.0, th, 0.0), a) for th in ths for a in (0, 1)]
    cases += [((x, 0.0, th, 0.0), a) for x in xs[:2] for th in ths[:2] for a in (0, 1)]
    return cases


@pytest.mark.parametrize("variant", [azo.DISCRETE, azo.CONTINUOUS])
def test_env_step_edges(variant):
    """azg_env_step at the env edges: == oracle bit for bit, and within 1e-13 of gym restated on math.sin / math.cos with equal
    terminal flags (Pendulum: the py_mod zero branch, |th| up to 1e5, actions +-2 and one f32 ulp around them, NaN, thdot landing
    on +-8; CartPole: x = +-2.4 and theta = +-12 deg, and one ulp inside and outside, with zero velocities)."""
    import enginelib as E
    cfg = azo.discrete_config() if variant == azo.DISCRETE else azo.continuous_config()
    if variant == azo.DISCRETE:
        cases = cartpole_edge_cases()
        s = np.array([c[0] for c in cases])
        a = np.array([c[1] for c in cases], np.float32)
    else:
        cases = pendulum_edge_cases()
        s = np.array([c[:2] for c in cases])
        a = np.array([c[2] for c in cases], np.float32)
    eng = E.SearchEngine(E.engine_config(cfg, 4))
    try:
        nxt, rew, term, obs = eng.env_step(s, a)
    finally:
        eng.close()
    cfg.math_mode = azo.MATH_DET
    ref = [azo.env_step(cfg, s[i], float(a[i])) for i in range(len(cases))]
    same = lambda x, y: np.array_equal(np.asarray(x), np.asarray(y), equal_nan=True)  # noqa: E731
    assert same(nxt, np.stack([r[0] for r in ref])) and same(rew, np.array([r[1] for r in ref]))
    assert np.array_equal(term.astype(bool), np.array([r[2] for r in ref]))
    assert same(obs, np.stack([r[3] for r in ref]))
    for i in range(len(cases)):
        st, rw, tm = gym_cartpole(tuple(s[i]), int(a[i])) if variant == azo.DISCRETE else gym_pendulum(s[i][0], s[i][1], a[i])
        assert bool(term[i]) == tm, (cases[i], tm)
        assert np.allclose(nxt[i], st, rtol=1e-13, atol=1e-13, equal_nan=True), (cases[i], nxt[i], st)
        assert np.allclose(rew[i], rw, rtol=1e-13, atol=1e-13, equal_nan=True), (cases[i], rew[i], rw)
    if variant == azo.DISCRETE:  # the inputs decide termination: exactly on the threshold is inside
        assert not term[:4].any() and term[4:6].all()

"""CPU side of the kernel matrix: the f64 bound (f64ref.py) holds for the oracle over the whole shape space the engine accepts,
the bound rejects a subtly wrong Q8 contract, every kernel instantiation in engine.cu has a case in the GPU matrix, and
EngineConfig.q8_supported() states the condition azg_create checks."""
import os
import re

import numpy as np
import pytest

from oracle import azo
import f64ref as F
import test_kernel_matrix_gpu as M

ENGINE_CU = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "alphazero_gym_b200", "csrc", "engine.cu")


def _shapes(variant):
    """Both variants x hidden {64, 128} x n_hidden 1-4 x six activations x K 1-8, in FP32, and in Q8 where the engine accepts it."""
    S = M.CARTPOLE if variant == azo.DISCRETE else M.PENDULUM
    for H in (64, 128):
        for L in (1, 2, 3, 4):
            for act in M.ACTS:
                for K in ((0,) if S == M.CARTPOLE else range(1, 9)):
                    for q8 in (False, True):
                        cfg = M.make_cfg(S, act, L, K, hidden=H, q8=q8)
                        if not q8 or M.q8_accepted(cfg):
                            yield cfg


@pytest.mark.parametrize("kind", ["default", "x10", "edge"])
@pytest.mark.parametrize("variant", [azo.DISCRETE, azo.CONTINUOUS])
def test_oracle_within_f64_bound(variant, kind):
    """V, raw head outputs and post-processed heads of the oracle lie within the derived bound of the f64 evaluation, for every
    shape, with default-initialised, x10 (trained-like) and edge weights (zero / 1e-30 / power-of-two rows)."""
    n = 0
    for cfg in _shapes(variant):
        w = M.weights(cfg, kind)
        x = M.observations(cfg, 48, seed=cfg.n_hidden + cfg.num_components)
        V, raw = azo.mlp_forward(cfg, w, x)
        post = np.stack([azo.head_post(cfg, r) for r in raw])
        ref = F.forward(cfg, w, x)
        for what, got, r, b in (("V", V, ref["V"], ref["bV"]), ("head", raw, ref["head"], ref["bhead"]),
                                ("post", post, ref["post"], ref["bpost"])):
            ok, ratio = F.within(got, r, b)
            assert ok, (f"H={cfg.hidden} L={cfg.n_hidden} act={cfg.activation} K={cfg.num_components} q8={cfg.eval_mode}: {what} "
                        f"outside the bound (worst ratio {ratio:.3g})")
        n += 1
    heads = 1 if variant == azo.DISCRETE else 8
    assert n == 2 * 4 * 6 * heads + 2 * 2 * min(heads, 5)  # FP32 shapes + Q8 shapes (relu / elu, 2 or 3 layers, K <= 5)


def _q8_cases():
    return [(S, act, L) for S in (M.CARTPOLE, M.PENDULUM) for act in (azo.ACT_RELU, azo.ACT_ELU) for L in (2, 3)]


def _layer_ratios(cfg, ref, V, raw, acts):
    r = [F.within(V, ref["V"], ref["bV"])[1], F.within(raw, ref["head"], ref["bhead"])[1]]
    return max(r + [F.within(a, ar, er)[1] for a, (ar, er) in zip(acts, ref["layers"])])


@pytest.mark.parametrize("S,act,L", _q8_cases())
def test_bound_discriminates_q8_contract(S, act, L):
    """The numpy restatement of the Q8 contract equals the oracle bit for bit and stays within the bound at every layer; the same
    contract without the PC digit products, or with one output's scale off by a factor of 2, leaves it."""
    cfg = M.make_cfg(S, act, L, 2, q8=True)
    w = M.weights(cfg, "x10")
    x = M.observations(cfg, 200, seed=L)[4:]  # rows in the environments' range
    ref = F.forward(cfg, w, x, trace=True)
    V, raw, acts = F.q8_contract(cfg, w, x)
    Vo, rawo = azo.mlp_forward(cfg, w, x)
    assert np.array_equal(V, Vo) and np.array_equal(raw, rawo)
    assert _layer_ratios(cfg, ref, V, raw, acts) <= 1.0
    assert _layer_ratios(cfg, ref, *F.q8_contract(cfg, w, x, drop_pc=True)) > 2.0
    assert _layer_ratios(cfg, ref, *F.q8_contract(cfg, w, x, scale_off=(1, 5))) > 100.0


def test_dispatch_tables_have_gpu_cases():
    """Every FUSED_CASE / QMLP_CASE / MLP_CASE instantiation in engine.cu has a case in the GPU matrix (and no case names a
    kernel that is not compiled)."""
    src = open(ENGINE_CU).read()

    def table(macro):
        calls = re.findall(r"\b" + macro + r"\((\d+), (\d+), (\d+)\)", src)
        return {tuple(int(v) for v in c) for c in calls}

    fused, qmlp, mlp = table("FUSED_CASE"), table("QMLP_CASE"), table("MLP_CASE")
    assert len(fused) == 8 and len(qmlp) == 8 and len(mlp) == 24
    assert fused == qmlp == set(M.QMLP_SHAPES)
    assert mlp == set(M.MLP_SHAPES)
    searched = {(S, a, nl) for S, a, nl, _, _ in M.SEARCH_CASES}
    assert searched == fused
    for S in (M.CARTPOLE, M.PENDULUM):
        kernels = {k for s, _, _, _, k in M.SEARCH_CASES if s == S}
        assert kernels == set(M.SEARCH_KERNELS[S])
    assert {K for S, _, _, K, _ in M.SEARCH_CASES if S == M.PENDULUM} == {1, 2, 3, 4}


def test_q8_supported_matches_engine_condition():
    """EngineConfig.q8_supported() against a restatement of azg_create's check (hidden 128, n_hidden 2 or 3, value + head padded
    to a multiple of 4 within 16 outputs, relu or elu), over every shape of the matrix."""
    import enginelib as E
    n = 0
    for variant in (azo.DISCRETE, azo.CONTINUOUS):
        for cfg in _shapes(variant):
            if cfg.eval_mode == azo.EVAL_Q8:
                continue
            assert E.engine_config(cfg, 1).q8_supported() == M.q8_accepted(cfg), (cfg.hidden, cfg.n_hidden, cfg.activation,
                                                                                   cfg.num_components)
            n += 1
    assert n == 2 * 4 * 6 * (1 + 8)

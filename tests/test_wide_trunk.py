"""CPU side of the hidden widths other than 64 / 128: the oracle's FP32 evaluation lies within the f64 bound (f64ref.py) for every
streamed width, depth, activation, input width and head; every k_mlp_stream instantiation in engine.cu has a case in
test_wide_trunk_gpu.py; the Python layer picks the FP32 per-simulation schedule for these widths and keeps refusing mixed ones."""
import os
import re

import numpy as np
import pytest

from oracle import azo
import f64ref as F
import test_kernel_matrix_gpu as M
import test_wide_trunk_gpu as W

ENGINE_CU = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "alphazero_gym_b200", "csrc", "engine.cu")


@pytest.mark.parametrize("kind", ["default", "x10", "edge"])
@pytest.mark.parametrize("env", sorted(W.ENVS))
def test_oracle_within_f64_bound(env, kind):
    """V, raw head outputs and post-processed heads of the oracle within the bound of the f64 evaluation, for hidden 32 ... 256,
    n_hidden 1-4, the six activations and every head size of the env."""
    n = 0
    S, heads = W.ENVS[env]
    for H in W.WIDTHS:
        for L in (1, 2, 3, 4):
            for act in W.ACTS:
                for K in heads:
                    cfg = W.make_cfg(env, act, L, K, hidden=H)
                    assert cfg.state_dim == S
                    w = M.weights(cfg, kind)
                    x = W.observations(cfg, 24, seed=L + K + H)
                    V, raw = azo.mlp_forward(cfg, w, x)
                    post = np.stack([azo.head_post(cfg, r) for r in raw])
                    ref = F.forward(cfg, w, x)
                    for what, got, r, b in (("V", V, ref["V"], ref["bV"]), ("head", raw, ref["head"], ref["bhead"]),
                                            ("post", post, ref["post"], ref["bpost"])):
                        ok, ratio = F.within(got, r, b)
                        assert ok, f"{env} H={H} L={L} act={act} K={K}: {what} outside the bound (worst ratio {ratio:.3g})"
                    n += 1
    assert n == len(W.WIDTHS) * 4 * 6 * len(heads)


def test_stream_dispatch_table_has_gpu_cases():
    """Every MLP_STREAM_CASE(S, ACT) of engine.cu has a case in the GPU matrix, and every case names a compiled kernel; the GPU
    matrix reaches every env of each input width."""
    src = open(ENGINE_CU).read()
    table = {tuple(int(v) for v in c) for c in re.findall(r"\bMLP_STREAM_CASE\((\d+), (\d+)\)", src)}
    assert len(table) == 24
    assert table == set(W.STREAM_SHAPES)
    assert {S for S, _ in W.ENVS.values()} == {S for S, _ in W.STREAM_SHAPES}


def test_rows_per_pass_fit_shared_memory():
    """The pass size the GPU tests mirror: at least 64 rows, at most 16 warps, and inside the shared memory of a B200 block for
    every width and head (at 256 wide, 128 rows per pass)."""
    for env, (S, heads) in W.ENVS.items():
        for H in W.WIDTHS:
            for K in heads:
                cfg = W.make_cfg(env, azo.ACT_RELU, 2, K, hidden=H)
                R = W.rows_per_pass(cfg)
                assert R >= 64 and (R // 64) * (H // 32) <= 16
                assert W.stream_smem(H, S, cfg.head_dim, R) <= W.SMEM_OPTIN, (env, H, K)
                if H == 256:
                    assert R == 128


def test_python_layer_at_wide_trunk():
    """EngineConfig at hidden 256 selects the FP32 evaluation and one launch per simulation; make_policy / describe_model carry
    a uniform 256-wide trunk and still refuse mixed widths."""
    from alphazero_gym_b200.engine import EngineConfig
    from alphazero_gym_b200._cabi import CONTINUOUS, DISCRETE
    from alphazero_gym_b200.network import describe_model, make_policy
    for variant, sd in ((DISCRETE, 4), (CONTINUOUS, 3)):
        for H in W.WIDTHS:
            cfg = EngineConfig(variant=variant, state_dim=sd, hidden=H, n_hidden=2)
            assert not cfg.q8_supported() and not cfg.is_q8() and not cfg.is_fused()
    d = describe_model(make_policy(4, 1, "discrete", [256, 256], "relu", num_actions=2))
    assert d["hidden"] == 256 and d["n_hidden"] == 2
    d = describe_model(make_policy(3, 1, "normal", [192, 192, 192], "elu", num_components=3, action_bound=2.0))
    assert d["hidden"] == 192 and d["n_hidden"] == 3 and d["head_dim"] == 9
    with pytest.raises(NotImplementedError):
        make_policy(4, 1, "discrete", [256, 128], "relu", num_actions=2)

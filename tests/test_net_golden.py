"""CPU suite: the fp32 network restatement (oracle/net_oracle.py) against tests/golden/net_*.npz - outputs of the
reference's own `build_model` functions traced under oracle/keras_shim.py (generator: oracle/gen_net_golden.py).
This pins the WIRING of the restatement (and the checkpoint names keras_bridge predicts) to the reference's source;
the layer arithmetic on both sides is PyTorch fp32, hence the tight tolerances (2e-5 = fp32 round-off through ten
blocks with differently associated BatchNorm affines; a wiring mistake shows up at 1e-2 and above)."""
import ast
import glob
import os

import numpy as np
import pytest
import torch

from grok_alpha_zero_b200 import keras_bridge, netspec
from net_oracle import NetOracle

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
FIXTURES = sorted(f for f in glob.glob(os.path.join(GOLD, "net_*.npz")) if "se_block" not in f)


def load_case(path):
    z = np.load(path)
    meta = ast.literal_eval(str(z["meta"]))
    spec = netspec.build_spec(meta["game"], meta["head"], **meta["over"])
    init = meta.get("init", dict(residual_gain=meta["residual_gain"]))     # "_g1" fixtures: undamped he_normal, fp32 kernels
    W = netspec.init_weights(spec, seed=meta["seed_w"], **init)
    return z, meta, spec, W


def test_fixture_inventory():
    assert len(FIXTURES) == 9
    assert {os.path.basename(f).split("_")[1] for f in FIXTURES} == {"gomoku", "connect4", "tictactoe"}


@pytest.mark.parametrize("path", FIXTURES, ids=lambda p: os.path.basename(p)[4:-4])
def test_restatement_matches_the_traced_reference_model(path):
    z, meta, spec, W = load_case(path)
    out = NetOracle(spec, W).forward(z["states"])
    # fp32 round-off scales with the magnitude of the activations: the undamped "_g1" fixtures reach |logit| ~ 150
    k = max(1.0, float(np.abs(z["logits"]).max()) / 8.0)
    np.testing.assert_allclose(out["logits"].numpy(), z["logits"], rtol=0, atol=2e-5 * k)
    np.testing.assert_allclose(out["value"].numpy().reshape(-1), z["value"], rtol=0, atol=2e-5 * k)
    np.testing.assert_allclose(out["policy"].numpy(), z["policy"], rtol=0, atol=(2e-6 if meta["head"] != "linear" else 2e-5) * k
                               if k == 1.0 else 2e-5 * k)      # a probability moves by at most 0.25 x its logit error
    if meta["head"] != "linear":
        np.testing.assert_allclose(z["policy"].sum(-1), 1.0, atol=1e-5)
    # dtype of the policy output as the builders declare it: float64 softmax for Gomoku / Connect4
    # (Gomoku/Build_Model.py:58, Connect4/Build_Model.py:57), float32 everywhere else
    want64 = meta["head"] == "softmax" and meta["game"] in ("gomoku", "connect4")
    assert str(z["policy_dtype"]) == ("float64" if want64 else "float32")


@pytest.mark.parametrize("path", FIXTURES, ids=lambda p: os.path.basename(p)[4:-4])
def test_checkpoint_names_are_the_traced_layer_names(path):
    z, meta, spec, W = load_case(path)
    predicted = set(keras_bridge.keras_layer_names(spec).values())
    assert predicted == set(str(n) for n in z["layer_names"])


def test_se_block_matches_the_reference_layer():
    z = np.load(os.path.join(GOLD, "net_se_block.npz"))
    W = {"b.se1.kernel": z["w1"], "b.se1.bias": z["b1"], "b.se2.kernel": z["w2"], "b.se2.bias": z["b2"]}
    x = torch.from_numpy(z["x"][:, 0]).permute(0, 3, 1, 2)                       # (B, 1, H, W, C) -> NCHW
    y = NetOracle(None, W).se(x, "b").permute(0, 2, 3, 1).numpy()
    np.testing.assert_allclose(y, z["y"][:, 0], rtol=0, atol=1e-6)

"""Backbone features without a GPU: the CPU reference of get_intermediate_layers (tests/features_ref.py) against what
the unmodified reference stored (tests/golden: norm_rows = model.dino(x)[:, rows], oracle/make_golden.py), and the
Python surface of model.dino on a CPU model (it raises: there is no CPU fallback)."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import GOLDEN_CASES, load_golden
from dino_b200 import DINOSeg, synthetic
from features_ref import feature_errors, intermediate_layers
from oracle import dinoseg_oracle as O


def _case(name):
    gd = load_golden(name)
    m = gd["meta"]
    cfg = synthetic.make_config(m["arch"], m["n_blocks"], m["n_classes"], head=m.get("head", "mlp"))
    sd = synthetic.init_state_dict(cfg, m["seed"], m["variant"])
    x = synthetic.make_frames(m["batch"], m["res"], m["seed"])
    return gd, m, cfg, sd, x


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_intermediate_layers_reproduce_the_reference_features(name):
    """The last element of get_intermediate_layers(x, n_blocks) is the reference's model.dino(x) at the stored rows, and
    every element is dino.norm applied to the residual stream after its block (O.backbone's stages)."""
    gd, m, cfg, sd, x = _case(name)
    torch.set_num_threads(max(1, min(8, os.cpu_count() or 1)))
    nb = cfg["n_blocks"]
    feats = intermediate_layers(sd, cfg, x, nb)
    assert len(feats) == nb
    stages = {}
    full = O.backbone(sd, cfg, x, stages=stages)
    assert torch.equal(feats[-1], full)
    got = feats[-1][:, gd["rows"]].numpy()
    assert got.shape == gd["norm_rows"].shape
    assert np.abs(got - gd["norm_rows"]).max() <= 1e-6 * max(1.0, float(np.abs(gd["norm_rows"]).max()))
    d = cfg["embed_dim"]
    for i, f in enumerate(feats):
        ref = F.layer_norm(stages[f"block{i}"], (d,), sd["dino.norm.weight"], sd["dino.norm.bias"], cfg["ln_eps"])
        assert torch.equal(f, ref), i
    # n counts back from the last block; n > n_blocks gives every block
    assert len(intermediate_layers(sd, cfg, x, 1)) == 1 and len(intermediate_layers(sd, cfg, x, nb + 2)) == nb


def test_feature_error_measures():
    ref = torch.randn(2, 5, 8, dtype=torch.float64)
    assert feature_errors(ref, ref) == (0.0, 0.0, pytest.approx(1.0))
    worse = ref.clone()
    worse[1, 3] = -worse[1, 3]
    rel, fro, cos = feature_errors(worse, ref)
    assert rel > 0 and fro > 0 and cos == pytest.approx(-1.0)


def test_backbone_features_on_a_cpu_model_raise():
    m = DINOSeg(head="mlp", n_blocks=2)
    x = torch.zeros(1, 3, 64, 64)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.dino(x)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.dino.get_intermediate_layers(x, n=2)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.features(x)
    for bad in (0, -1, 1.5, "2"):
        with pytest.raises(ValueError):
            m.dino.get_intermediate_layers(x, n=bad)
    # the state dict is the reference's: the backbone's forward adds no parameter or buffer
    ref = synthetic.init_state_dict(synthetic.make_config("vit_small", 2, 7))
    assert sorted(m.state_dict()) == sorted(ref)

"""Image embeddings without a GPU: the CLS-only restatement of the last block (tests/embeddings_ref.py) against row 0 of
the oracle's full block on the golden cases, upstream's embedding expressions on the stored reference features, and
the Python surface of DINOSeg.embeddings on a CPU model (it raises: there is no CPU fallback)."""
import os

import pytest
import torch
import torch.nn.functional as F

from conftest import GOLDEN_CASES, load_golden
from dino_b200 import DINOSeg, synthetic
import embeddings_ref as E
from features_ref import intermediate_layers
from oracle import dinoseg_oracle as O


def _case(name):
    gd = load_golden(name)
    m = gd["meta"]
    cfg = synthetic.make_config(m["arch"], m["n_blocks"], m["n_classes"], head=m.get("head", "mlp"))
    sd = synthetic.init_state_dict(cfg, m["seed"], m["variant"])
    x = synthetic.make_frames(m["batch"], m["res"], m["seed"])
    return gd, m, cfg, sd, x


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_cls_only_block_equals_row_0_of_the_full_block(name):
    """The last block restated for the CLS row (LayerNorm1 and K / V over every row, q of row 0, proj and MLP on one
    row) gives row 0 of the oracle's full block to fp32 rounding, and the embedding built on it is the stored
    reference's CLS embedding (norm_rows[:, 0], rows[0] == 0)."""
    gd, m, cfg, sd, x = _case(name)
    torch.set_num_threads(max(1, min(8, os.cpu_count() or 1)))
    nb, heads, eps = cfg["n_blocks"], cfg["num_heads"], cfg["ln_eps"]
    t = O.prepare_tokens(sd, x)
    for i in range(nb - 1):
        t = O.block(sd, i, t, heads, eps)
    full = O.block(sd, nb - 1, t, heads, eps)[:, 0]
    row = E.cls_block(sd, nb - 1, t, heads, eps)
    scale = float(full.abs().max())
    assert float((row - full).abs().max()) <= 2e-6 * scale, float((row - full).abs().max()) / scale
    assert int(gd["rows"][0]) == 0
    emb = E.cls_embedding_shortcut(sd, cfg, x)
    ref = torch.from_numpy(gd["norm_rows"][:, 0])
    assert float((emb - ref).abs().max()) <= 1e-5 * max(1.0, float(ref.abs().max()))


@pytest.mark.parametrize("name", ["s8_nb3_240_b2_trained", "b8_nb4_240_refinit", "s8_nb1_64_trained"])
def test_upstream_expressions(name):
    """from_layers is upstream's torch.cat of the CLS rows (oldest block first), and its avgpool form interleaves the
    last CLS row with the patch-token mean."""
    gd, m, cfg, sd, x = _case(name)
    nb, d, b = cfg["n_blocks"], cfg["embed_dim"], m["batch"]
    layers = intermediate_layers(sd, cfg, x, nb)
    cat = E.from_layers(layers)
    assert cat.shape == (b, nb * d)
    for k in range(nb):
        assert torch.equal(cat[:, k * d:(k + 1) * d], layers[k][:, 0])
    pooled = E.from_layers(layers[-1:], avgpool=True)
    assert pooled.shape == (b, 2 * d)
    assert torch.equal(pooled[:, 0::2], layers[-1][:, 0])
    assert torch.equal(pooled[:, 1::2], layers[-1][:, 1:].mean(1))
    assert torch.equal(E.embeddings(sd, cfg, x, 1), layers[-1][:, 0])
    assert torch.equal(E.embeddings(sd, cfg, x, nb + 1), cat)


def test_rectangular_shortcut_matches_the_full_block():
    """The shortcut on a 48 x 64 frame (rect_ref's tokens) against row 0 of the full last block."""
    cfg = synthetic.make_config("vit_small", 2, 7)
    sd = synthetic.init_state_dict(cfg, 3, "trained_like")
    x = torch.randn(2, 3, 48, 64, generator=torch.Generator().manual_seed(0))
    full = E.embeddings(sd, cfg, x, 1)
    short = E.cls_embedding_shortcut(sd, cfg, x)
    assert full.shape == short.shape == (2, 384)
    assert float((full - short).abs().max()) <= 2e-5 * float(full.abs().max())


def test_embeddings_on_a_cpu_model_raise():
    m = DINOSeg(head="mlp", n_blocks=2)
    x = torch.zeros(1, 3, 64, 64)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.embeddings(x)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.embeddings(x, 2)
    for bad in (0, -1, 1.5, "2"):
        with pytest.raises(ValueError):
            m.embeddings(x, n=bad)
    for n in (2, 3):
        with pytest.raises(ValueError, match="avgpool"):
            m.embeddings(x, n=n, avgpool=True)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.embeddings(x, n=1, avgpool=True)

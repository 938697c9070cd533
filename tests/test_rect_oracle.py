"""The CPU reference for non-square frames (tests/rect_ref.py: H x W, both multiples of 8): the positional table
resampled per axis, the token layout and the uint8 resize to (H, W), and its agreement with the golden-pinned oracle on
square frames.  The GPU path is pinned to it in tests/test_gpu_rect.py.

The reference (vision_transformer.py:202-235) names x.shape[2] `w`, so its first scale factor applies to the rows:
scale_factor = ((gh + 0.1) / G0, (gw + 0.1) / G0) for a gh x gw patch grid.  The table is used unchanged only for
gh == gw == G0 (`npatch == N and w == h`): a 14 x 56 grid has 784 patches like 28 x 28 and is still resampled.
"""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import rect_ref as R
from dino_b200 import synthetic
from oracle import dinoseg_oracle as O
from oracle import preproc_oracle as P

GRIDS = [(60, 80), (80, 60), (14, 56), (1, 8), (8, 1), (28, 28)]


@pytest.mark.parametrize("gh,gw", GRIDS)
def test_bicubic_numpy_restatement_matches_torch_rect(gh, gw):
    """Same bar as the square test in test_oracle_golden.py (fp32 summation order differs)."""
    torch.manual_seed(gh * 1000 + gw)
    pos = torch.randn(1, 785, 48)
    ref = R.interpolate_pos_encoding(pos, gh, gw)[0].numpy()
    got = R.bicubic_pos_table_numpy(pos[0].numpy(), gh, gw)
    assert got.shape == ref.shape == (gh * gw + 1, 48)
    assert np.abs(got - ref).max() <= 2e-5
    if (gh, gw) == (28, 28):
        assert np.array_equal(ref, pos[0].numpy()) and np.array_equal(got, pos[0].numpy())


def test_rect_table_follows_the_reference_call():
    """interpolate_pos_encoding(pos, gh, gw) is the reference's F.interpolate call on a [B,3,8*gh,8*gw] input, with
    (gh + 0.1) / G0 for the rows; the transposed grid is a different table; the square form is unchanged."""
    torch.manual_seed(3)
    pos = torch.randn(1, 785, 16)
    gh, gw = 60, 80
    w0, h0 = gh + 0.1, gw + 0.1
    grid = pos[:, 1:].reshape(1, 28, 28, 16).permute(0, 3, 1, 2)
    ref = F.interpolate(grid, scale_factor=(w0 / math.sqrt(784), h0 / math.sqrt(784)), mode="bicubic")
    assert tuple(ref.shape[-2:]) == (gh, gw)
    ref = torch.cat((pos[:, :1], ref.permute(0, 2, 3, 1).reshape(1, -1, 16)), dim=1)
    got = R.interpolate_pos_encoding(pos, gh, gw)
    assert torch.equal(got, ref)
    assert not torch.equal(R.interpolate_pos_encoding(pos, gw, gh), got)
    assert torch.equal(O.interpolate_pos_encoding(pos, 30), R.interpolate_pos_encoding(pos, 30, 30))


def test_identity_needs_a_square_grid():
    """14 x 56 has G0 * G0 patches but is not the identity (reference condition `npatch == N and w == h`)."""
    torch.manual_seed(1)
    pos = torch.randn(1, 785, 8)
    assert R.interpolate_pos_encoding(pos, 28, 28) is pos
    t = R.interpolate_pos_encoding(pos, 14, 56)
    assert t.shape == (1, 785, 8) and not torch.equal(t, pos)


def test_prepare_tokens_rect():
    """Rectangular frames: CLS then the gh*gw patches row by row, each plus its entry of the gh x gw table."""
    torch.manual_seed(0)
    d = 16
    sd = {"dino.patch_embed.proj.weight": torch.randn(d, 3, 8, 8), "dino.patch_embed.proj.bias": torch.randn(d),
          "dino.cls_token": torch.randn(1, 1, d), "dino.pos_embed": torch.randn(1, 785, d)}
    x = torch.randn(2, 3, 48, 80)
    t = R.prepare_tokens(sd, x)
    assert t.shape == (2, 1 + 6 * 10, d)
    pos = R.interpolate_pos_encoding(sd["dino.pos_embed"], 6, 10)
    i, j = 4, 7
    patch = x[:, :, 8 * i:8 * i + 8, 8 * j:8 * j + 8]
    emb = (patch[:, None] * sd["dino.patch_embed.proj.weight"][None]).sum((2, 3, 4)) + sd["dino.patch_embed.proj.bias"]
    assert torch.allclose(t[:, 1 + i * 10 + j], emb + pos[0, 1 + i * 10 + j], atol=1e-4)


@pytest.mark.parametrize("src,dst", [((480, 640), (240, 320)),     # downscale
                                     ((120, 160), (480, 640)),     # upscale
                                     ((480, 640), (640, 480)),     # up on one axis, down on the other
                                     ((300, 200), (112, 448)),
                                     ((123, 77), (64, 8)),
                                     ((480, 640), (480, 640))])    # same size: passes through
def test_resize_linear_u8_rect_matches_cv2(src, dst):
    import cv2
    rng = np.random.default_rng(src[0] * 31 + dst[1])
    img = rng.integers(0, 256, (src[0], src[1], 3), dtype=np.uint8)
    ref = cv2.resize(img, (dst[1], dst[0]), interpolation=cv2.INTER_LINEAR)
    got = R.resize_linear_u8(img, dst)
    assert got.shape == (dst[0], dst[1], 3)
    assert np.array_equal(got, ref)
    x = R.preprocess(img, dst)
    assert x.shape == (3, dst[0], dst[1]) and x.dtype == np.float32


def test_resize_square_forms_agree():
    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, (360, 500, 3), dtype=np.uint8)
    assert np.array_equal(P.resize_linear_u8(img, 240), R.resize_linear_u8(img, (240, 240)))
    assert np.array_equal(P.preprocess(img, 240), R.preprocess(img, (240, 240)))


@pytest.mark.parametrize("g", [8, 28, 30, 60])
def test_square_tables_equal_the_oracle(g):
    """On square grids the rectangular reference is the golden-pinned oracle: same table, bit for bit."""
    torch.manual_seed(g)
    pos = torch.randn(1, 785, 48)
    assert torch.equal(R.interpolate_pos_encoding(pos, g, g), O.interpolate_pos_encoding(pos, g))
    assert np.array_equal(R.bicubic_pos_table_numpy(pos[0].numpy(), g, g), O.bicubic_pos_table_numpy(pos[0].numpy(), g))


@pytest.mark.parametrize("arch,nb,head,res,batch", [("vit_small", 2, "mlp", 64, 2), ("vit_small", 1, "linear", 40, 1),
                                                    ("vit_base", 1, "mlp", 224, 1)])
def test_square_frames_equal_the_oracle(arch, nb, head, res, batch):
    """Log-probs, features and CLS attention of the rectangular reference on square frames equal the oracle's bit for
    bit (the oracle is pinned to the reference's own outputs by tests/golden)."""
    cfg = synthetic.make_config(arch, nb, 7, head=head)
    sd = synthetic.init_state_dict(cfg, 4, "trained_like")
    x = synthetic.make_frames(batch, res, seed=2)
    assert torch.equal(R.forward(sd, cfg, x), O.forward(sd, cfg, x))
    assert torch.equal(R.intermediate_layers(sd, cfg, x, 1)[-1], O.backbone(sd, cfg, x))
    assert torch.equal(R.last_selfattention_cls(sd, cfg, x), O.last_selfattention_cls(sd, cfg, x))

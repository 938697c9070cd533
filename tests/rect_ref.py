"""CPU reference for non-square frames (test infrastructure): the reference's prepare_tokens / interpolate_pos_encoding
(vision_transformer.py:202-235) on [B,3,H,W] input, restated on top of the oracle's block and head
(oracle/dinoseg_oracle.py), and the uint8 resize to (H, W) on top of the preprocessing oracle's OpenCV coefficients
(oracle/preproc_oracle.py).

Axis convention: the reference writes `B, nc, w, h = x.shape`, so its `w` is the ROW count and the first scale factor
(w0 / sqrt(N)) of its F.interpolate call applies to the rows: scale_factor = ((gh + 0.1) / G0, (gw + 0.1) / G0) for a
gh x gw patch grid.  The table is returned unchanged only for `npatch == N and w == h`, i.e. gh == gw == G0.

There is no copy of the reference here to produce rectangular goldens, so rectangular parity rests on this module.
It calls the same F.conv2d and F.interpolate(mode='bicubic') the reference calls, and on square frames it reproduces
the golden-pinned oracle bit for bit (tests/test_rect_oracle.py).
"""
import math

import numpy as np
import torch
import torch.nn.functional as F

from oracle import dinoseg_oracle as O
from oracle import preproc_oracle as P


def interpolate_pos_encoding(pos_embed: torch.Tensor, gh: int, gw: int) -> torch.Tensor:
    """vision_transformer.py:202-222 for a gh x gw patch grid (gh rows). pos_embed: [1, G0*G0+1, D]."""
    n_src = pos_embed.shape[1] - 1
    g0 = int(math.sqrt(n_src))
    if gh * gw == n_src and gh == gw:                    # :205-206 (npatch == N and w == h)
        return pos_embed
    dim = pos_embed.shape[-1]
    w0, h0 = gh + 0.1, gw + 0.1                          # :212-214 (w = rows)
    patch_pos = F.interpolate(
        pos_embed[:, 1:].reshape(1, g0, g0, dim).permute(0, 3, 1, 2),
        scale_factor=(w0 / math.sqrt(n_src), h0 / math.sqrt(n_src)),
        mode="bicubic",
    )
    assert int(w0) == patch_pos.shape[-2] and int(h0) == patch_pos.shape[-1]   # :220
    patch_pos = patch_pos.permute(0, 2, 3, 1).reshape(1, -1, dim)
    return torch.cat((pos_embed[:, 0].unsqueeze(0), patch_pos), dim=1)


def _bicubic_taps(g: int, g0: int):
    """Weights [g, 4] and clamped source indices [g, 4] of one axis resampled from g0 to g points."""
    rscale = np.float32(1.0 / ((g + 0.1) / float(g0)))
    src = rscale * (np.arange(g, dtype=np.float32) + np.float32(0.5)) - np.float32(0.5)
    i0 = np.minimum(np.floor(src).astype(np.int64), g0 - 1)
    t = np.clip(src - i0.astype(np.float32), 0, 1).astype(np.float32)
    return O._cubic_coeffs(t), np.clip(i0[:, None] + np.arange(-1, 3)[None, :], 0, g0 - 1)


def bicubic_pos_table_numpy(pos_embed: np.ndarray, gh: int, gw: int) -> np.ndarray:
    """Independent numpy restatement of the table above: [G0*G0+1, D] -> [gh*gw+1, D].  Per axis src =
    rscale*(dst+0.5)-0.5 with rscale = float32(1/scale_factor), taps floor(src)-1..+2 clamped to [0, G0-1], cubic
    weights with A = -0.75; x taps summed first, then y."""
    pos_embed = np.asarray(pos_embed, dtype=np.float32)
    n_src = pos_embed.shape[0] - 1
    g0 = int(math.sqrt(n_src))
    if gh * gw == n_src and gh == gw:
        return pos_embed.copy()
    d = pos_embed.shape[1]
    grid = pos_embed[1:].reshape(g0, g0, d)
    wy, iy = _bicubic_taps(gh, g0)
    wx, ix = _bicubic_taps(gw, g0)
    tmp = np.zeros((g0, gw, d), dtype=np.float32)
    for b in range(4):
        tmp += wx[None, :, b, None] * grid[:, ix[:, b], :]
    out = np.zeros((gh, gw, d), dtype=np.float32)
    for a in range(4):
        out += wy[:, a, None, None] * tmp[iy[:, a], :, :]
    return np.concatenate([pos_embed[:1], out.reshape(gh * gw, d)], axis=0)


def prepare_tokens(sd: dict, x: torch.Tensor) -> torch.Tensor:
    """vision_transformer.py:224-235 for [B,3,H,W]: CLS, then the patches row by row, plus the gh x gw table."""
    b, _, w, h = x.shape                                 # reference naming: w = rows, h = columns
    assert w % 8 == 0 and h % 8 == 0
    t = F.conv2d(x, sd["dino.patch_embed.proj.weight"], sd["dino.patch_embed.proj.bias"], stride=8)
    t = t.flatten(2).transpose(1, 2)
    t = torch.cat((sd["dino.cls_token"].expand(b, -1, -1), t), dim=1)
    return t + interpolate_pos_encoding(sd["dino.pos_embed"], w // 8, h // 8)


@torch.no_grad()
def intermediate_layers(sd: dict, cfg: dict, x: torch.Tensor, n: int = 1) -> list:
    """get_intermediate_layers (vision_transformer.py:282-290): dino.norm of the residual stream after each of the last
    n blocks, oldest first; the last element is VisionTransformer.forward for all tokens."""
    t = prepare_tokens(sd, x)
    nb = cfg["n_blocks"]
    d = t.shape[-1]
    out = []
    for i in range(nb):
        t = O.block(sd, i, t, cfg["num_heads"], cfg["ln_eps"])
        if nb - i <= n:
            out.append(F.layer_norm(t, (d,), sd["dino.norm.weight"], sd["dino.norm.bias"], cfg["ln_eps"]))
    return out


@torch.no_grad()
def forward(sd: dict, cfg: dict, x: torch.Tensor) -> torch.Tensor:
    """DINOSeg.forward (pl_torch_modules.py:239-256): [B,3,H,W] -> log-probs [B*gh*gw, C], one frame at a time."""
    outs = []
    for s in range(x.shape[0]):
        t = intermediate_layers(sd, cfg, x[s:s + 1], 1)[-1][:, 1:]
        outs.append(O.head(sd, t.reshape((-1, t.shape[-1]))))
    return torch.cat(outs, dim=0)


@torch.no_grad()
def last_selfattention_cls(sd: dict, cfg: dict, x: torch.Tensor) -> torch.Tensor:
    """Row 0 (CLS query) of get_last_selfattention (vision_transformer.py:273-280): [B, heads, N]."""
    t = prepare_tokens(sd, x)
    nb = cfg["n_blocks"]
    for i in range(nb - 1):
        t = O.block(sd, i, t, cfg["num_heads"], cfg["ln_eps"])
    p = f"dino.blocks.{nb - 1}."
    y = F.layer_norm(t, (t.shape[-1],), sd[p + "norm1.weight"], sd[p + "norm1.bias"], cfg["ln_eps"])
    _, attn = O.attention(sd, p + "attn.", y, cfg["num_heads"], return_attn=True)
    return attn[:, :, 0, :]


def resize_linear_u8(img: np.ndarray, hw) -> np.ndarray:
    """cv2.resize(img, (W, H), interpolation=cv2.INTER_LINEAR) for uint8 HWC images, one scale per axis."""
    oh, ow = hw
    h, w, _ = img.shape
    if h == oh and w == ow:
        return img.copy()
    x0, x1, a0, a1 = P._coef(ow, w, True)
    y0, y1, b0, b1 = P._coef(oh, h, False)
    im = img.astype(np.int64)
    rows0 = im[y0][:, x0] * a0[None, :, None] + im[y0][:, x1] * a1[None, :, None]
    rows1 = im[y1][:, x0] * a0[None, :, None] + im[y1][:, x1] * a1[None, :, None]
    out = (((b0[:, None, None] * (rows0 >> 4)) >> 16) + ((b1[:, None, None] * (rows1 >> 4)) >> 16) + 2) >> 2
    return np.clip(out, 0, 255).astype(np.uint8)


def preprocess(img_u8: np.ndarray, hw) -> np.ndarray:
    """uint8 HWC -> float32 CHW [3, H, W] as the reference's transforms produce it (Resize to (H, W), Normalize)."""
    x = resize_linear_u8(img_u8, hw).astype(np.float32)
    x -= np.array(P.IMAGENET_MEAN, dtype=np.float32) * np.float32(255.0)
    x *= np.reciprocal(np.array(P.IMAGENET_STD, dtype=np.float32) * np.float32(255.0))
    return np.ascontiguousarray(x.transpose(2, 0, 1))

"""CPU reference of the image embeddings (test infrastructure): upstream DINO's two embedding expressions applied to the
intermediate layers of features_ref / rect_ref, and a restatement of the last block for the CLS row alone - the
shortcut DINOSeg.embeddings takes on the GPU when it needs no patch mean.

Upstream (facebookresearch/dino):
- eval_knn / `model(x)`: the CLS token after the final norm, x[:, 0];
- eval_linear: torch.cat([x[:, 0] for x in model.get_intermediate_layers(inp, n)], dim=-1), and with avgpool
  torch.cat((output.unsqueeze(-1), torch.mean(intermediate_output[-1][:, 1:], dim=1).unsqueeze(-1)), dim=-1)
  followed by output.reshape(output.shape[0], -1).
"""
import torch
import torch.nn.functional as F

import features_ref
import rect_ref
from oracle import dinoseg_oracle as O


def from_layers(layers, avgpool=False):
    """Upstream's embedding of a list of normed token tensors [B, N, D] (oldest block first)."""
    out = torch.cat([t[:, 0] for t in layers], dim=-1)
    if avgpool:
        out = torch.cat((out.unsqueeze(-1), torch.mean(layers[-1][:, 1:], dim=1).unsqueeze(-1)), dim=-1)
        out = out.reshape(out.shape[0], -1)
    return out


@torch.no_grad()
def intermediate_layers(sd, cfg, x, n=1):
    """features_ref.intermediate_layers for square frames, rect_ref's restatement for [B,3,H,W] with H != W."""
    if x.shape[2] == x.shape[3]:
        return features_ref.intermediate_layers(sd, cfg, x, n)
    return rect_ref.intermediate_layers(sd, cfg, x, n)


@torch.no_grad()
def embeddings(sd, cfg, x, n=1, avgpool=False):
    """DINOSeg.embeddings(x, n, avgpool) in fp32 on the CPU."""
    return from_layers(intermediate_layers(sd, cfg, x, n), avgpool)


def _bf16(t):
    return t.to(torch.bfloat16).float()


@torch.no_grad()
def cls_block(sd, i, t, num_heads, eps, bf16_qkv=False):
    """Block i (vision_transformer.py:122-140) for the CLS row only: LayerNorm1 and the keys / values over every row,
    the query of row 0, then proj and the MLP on that one row.  t: [B, N, D] -> the block's output row 0, [B, D].
    bf16_qkv: round LayerNorm1's output, the qkv weight and the GEMM's q (pre-scaled by dh^-0.5 * log2(e)), k and v to
    bf16 as the GPU's qkv GEMM does, and take the softmax in log2 units; the rest stays fp32."""
    p = f"dino.blocks.{i}."
    b, n, d = t.shape
    hd = d // num_heads
    y = F.layer_norm(t, (d,), sd[p + "norm1.weight"], sd[p + "norm1.bias"], eps)
    w, bias = sd[p + "attn.qkv.weight"], sd[p + "attn.qkv.bias"]
    if bf16_qkv:
        y, w = _bf16(y), _bf16(w)
    q = F.linear(y[:, 0], w[:d], bias[:d]).reshape(b, num_heads, 1, hd)
    k = F.linear(y, w[d:2 * d], bias[d:2 * d]).reshape(b, n, num_heads, hd).transpose(1, 2)
    v = F.linear(y, w[2 * d:], bias[2 * d:]).reshape(b, n, num_heads, hd).transpose(1, 2)
    if bf16_qkv:
        log2e = 1.4426950408889634
        q, k, v = _bf16(q * (hd ** -0.5 * log2e)), _bf16(k), _bf16(v)
        attn = ((q @ k.transpose(-2, -1)) / log2e).softmax(dim=-1)
    else:
        attn = ((q @ k.transpose(-2, -1)) * (hd ** -0.5)).softmax(dim=-1)
    o = (attn @ v).reshape(b, d)
    x0 = t[:, 0] + F.linear(o, sd[p + "attn.proj.weight"], sd[p + "attn.proj.bias"])
    z = F.layer_norm(x0, (d,), sd[p + "norm2.weight"], sd[p + "norm2.bias"], eps)
    z = F.gelu(F.linear(z, sd[p + "mlp.fc1.weight"], sd[p + "mlp.fc1.bias"]))
    return x0 + F.linear(z, sd[p + "mlp.fc2.weight"], sd[p + "mlp.fc2.bias"])


@torch.no_grad()
def cls_embedding_shortcut(sd, cfg, x, bf16_qkv=False):
    """embeddings(x, 1) computed the way the GPU's CLS-only tail does: every block but the last in full, the last one
    for the CLS row only (cls_block), then the final norm.  [B, D]."""
    t = O.prepare_tokens(sd, x) if x.shape[2] == x.shape[3] else rect_ref.prepare_tokens(sd, x)
    nb = cfg["n_blocks"]
    for i in range(nb - 1):
        t = O.block(sd, i, t, cfg["num_heads"], cfg["ln_eps"])
    row = cls_block(sd, nb - 1, t, cfg["num_heads"], cfg["ln_eps"], bf16_qkv)
    return F.layer_norm(row, (row.shape[-1],), sd["dino.norm.weight"], sd["dino.norm.bias"], cfg["ln_eps"])

"""CPU reference of the backbone features (test infrastructure): VisionTransformer.get_intermediate_layers
(vision_transformer.py:282-290) restated on the oracle's prepare_tokens / block, and the error measures the feature
tests judge the GPU path by."""
import torch
import torch.nn.functional as F

from oracle import dinoseg_oracle as O

# bars for the GPU features against fp32 (bf16 GEMM / attention operands; the CPU emulation of that rounding reaches
# 2.3e-3 / 3.4e-3 max-abs-over-max for 'reference_init' ViT-S / ViT-B and 1.46e-2 for the 'trained_like' stress weights)
MAX_REL = {"reference_init": 1e-2, "trained_like": 4e-2}
FRO_REL = 2.5e-2
MIN_COS = 0.999


@torch.no_grad()
def intermediate_layers(sd, cfg, x, n=1):
    """The final norm (dino.norm) of the residual stream after each of the last n blocks, oldest first, as the reference
    loop `if len(self.blocks) - i <= n: output.append(self.norm(x))` computes it.  The last element is O.backbone()."""
    t = O.prepare_tokens(sd, x)
    nb = cfg["n_blocks"]
    d = t.shape[-1]
    out = []
    for i in range(nb):
        t = O.block(sd, i, t, cfg["num_heads"], cfg["ln_eps"])
        if nb - i <= n:
            out.append(F.layer_norm(t, (d,), sd["dino.norm.weight"], sd["dino.norm.bias"], cfg["ln_eps"]))
    return out


def feature_errors(got, ref):
    """-> (max-abs error / max |ref|, Frobenius error / Frobenius norm of ref, smallest per-token cosine similarity)."""
    got, ref = torch.as_tensor(got).double(), torch.as_tensor(ref).double()
    err = got - ref
    return (float(err.abs().max() / ref.abs().max()), float(err.norm() / ref.norm()),
            float(F.cosine_similarity(got, ref, dim=-1).min()))

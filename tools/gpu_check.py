#!/usr/bin/env python
"""Kernel-level bring-up checks for libdinoseg.so on a real B200.

Each check runs in its OWN subprocess (a device-side trap kills the CUDA context, so one
failing kernel must not take the other checks with it) under a timeout.  The references
are plain fp32 torch ops on the same GPU.

    python tools/gpu_check.py            # run everything, print a summary, exit 1 on failure
    python tools/gpu_check.py gemm_qkv   # run one check in-process
"""
from __future__ import annotations

import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _imports():
    import torch
    from dino_b200 import _lib
    return torch, _lib, _lib.load()


def _ptr(t):
    return t.data_ptr() if t is not None else None


def _report(name, ok, **kw):
    print("CHECK " + json.dumps({"name": name, "ok": bool(ok), **kw}), flush=True)
    return bool(ok)


# ------------------------------------------------------------------------------------------
def check_gemm(name, M, N, K, epi, with_bias=True, P=0, Ntok=0):
    torch, L, lib = _imports()
    torch.manual_seed(1)
    dev = "cuda"
    A = (torch.randn(M, K, device=dev) * 1.0).to(torch.bfloat16)
    W = (torch.randn(N, K, device=dev) * 0.05).to(torch.bfloat16)
    bias = torch.randn(N, device=dev) * 0.1 if with_bias else None
    ref = A.float() @ W.float().t()
    if bias is not None:
        ref = ref + bias
    pos = None
    if epi == L.EPI_BF16:
        scale_cols = N // 3
        ref[:, :scale_cols] *= 0.125
        out = torch.zeros(M, N, device=dev, dtype=torch.bfloat16)
        ldo = N
    elif epi == L.EPI_GELU_BF16:
        scale_cols = 0
        ref = torch.nn.functional.gelu(ref)
        out = torch.zeros(M, N, device=dev, dtype=torch.bfloat16)
        ldo = N
    elif epi == L.EPI_RESID_F32:
        scale_cols = 0
        out = torch.randn(M, N, device=dev)
        ref = ref + out
        ldo = N
    elif epi == L.EPI_PATCH_F32:
        scale_cols = 0
        assert M % P == 0
        B = M // P
        pos = torch.randn(Ntok, N, device=dev)
        out = torch.full((B * Ntok, N), 7.0, device=dev)
        full = torch.full((B, Ntok, N), 7.0, device=dev)
        full[:, 1:, :] = ref.view(B, P, N) + pos[1:].unsqueeze(0)
        ref = full.view(B * Ntok, N)
        ldo = N
    elif epi == L.EPI_RELU_F32:
        scale_cols = 0
        ref = torch.relu(ref)
        out = torch.zeros(M, N, device=dev)
        ldo = N
    rc = lib.dinoseg_op_gemm(_ptr(A), _ptr(W), _ptr(bias), _ptr(out), M, N, K, ldo, epi, 0.125, scale_cols,
                             _ptr(pos), P, Ntok, None)
    torch.cuda.synchronize()
    got = out.float()
    err = (got - ref).abs().max().item()
    scale = ref.abs().max().item()
    tol = 2e-2 * scale if out.dtype == torch.bfloat16 else 2e-3 * scale
    # locate the first bad element to help debugging layout bugs
    bad = ((got - ref).abs() > tol).nonzero()
    first_bad = bad[0].tolist() if bad.numel() else None
    return _report(name, rc == 0 and err <= tol, rc=rc, max_abs_err=err, ref_absmax=scale, tol=tol,
                   n_bad=int(bad.shape[0]), first_bad=first_bad)


def check_gemm_pair(name, M, N, K, epi=0):
    """GEMM run by CTA pairs (cta_group::2) vs fp32 torch on the same bf16 operands, and bit-identical to the
    single-CTA kernel (same MMAs per output row, same epilogue).  epi: 0 bf16 (q scaled), 1 GELU bf16, 2 residual fp32."""
    torch, L, lib = _imports()
    torch.manual_seed(1)
    dev = "cuda"
    A = (torch.randn(M, K, device=dev) * 1.0).to(torch.bfloat16)
    W = (torch.randn(N, K, device=dev) * 0.05).to(torch.bfloat16)
    bias = torch.randn(N, device=dev) * 0.1
    ref = A.float() @ W.float().t() + bias
    scale_cols = 0
    if epi == L.EPI_BF16:
        scale_cols = N // 3
        ref[:, :scale_cols] *= 0.125
        out = torch.zeros(M, N, device=dev, dtype=torch.bfloat16)
    elif epi == L.EPI_GELU_BF16:
        ref = torch.nn.functional.gelu(ref)
        out = torch.zeros(M, N, device=dev, dtype=torch.bfloat16)
    else:
        out = torch.randn(M, N, device=dev)
        ref = ref + out
    one = out.clone()
    rc = lib.dinoseg_op_gemm_pair(_ptr(A), _ptr(W), _ptr(bias), _ptr(out), M, N, K, N, epi, 0.125, scale_cols, None)
    rc1 = lib.dinoseg_op_gemm(_ptr(A), _ptr(W), _ptr(bias), _ptr(one), M, N, K, N, epi, 0.125, scale_cols, None, 0, 0, None)
    torch.cuda.synchronize()
    err = (out.float() - ref).abs().max().item()
    scale = ref.abs().max().item()
    tol = (2e-2 if out.dtype == torch.bfloat16 else 2e-3) * scale
    same = bool(torch.equal(out, one))
    bad = ((out.float() - ref).abs() > tol).nonzero()
    return _report(name, rc == 0 and rc1 == 0 and err <= tol and same, rc=rc, max_abs_err=err, ref_absmax=scale, tol=tol,
                   identical_to_single_cta=same, n_bad=int(bad.shape[0]), first_bad=bad[0].tolist() if bad.numel() else None)


def check_attention(name, B, N, H, spread=1.0, shift=0.0, redone=0):
    torch, L, lib = _imports()
    torch.manual_seed(2)
    dev = "cuda"
    D = H * 64
    qkv = torch.randn(B, N, 3 * D, device=dev)
    qkv[..., :D] *= 0.125 * 2.0 * spread  # pre-scaled q (dh^-0.5 * log2 e folded in) with more spread than unit variance
    qkv[..., D:2 * D] += shift                 # a common offset of the keys moves whole rows of scores
    qkv = qkv.to(torch.bfloat16)
    out = torch.zeros(B * N, D, device=dev, dtype=torch.bfloat16)
    rc = lib.dinoseg_op_attention(_ptr(qkv), _ptr(out), B, N, H, None)
    torch.cuda.synchronize()
    # which kernel produced the result: the one without row maxima, or (scores out of its range) the classic one as its redo
    was_redone = lib.dinoseg_debug_attn_redone() if os.environ.get("DINOSEG_ATTN_UNSHIFTED", "1") != "0" else redone
    f = qkv.float().view(B, N, 3, H, 64).permute(2, 0, 3, 1, 4)
    q, k, v = f[0], f[1], f[2]
    ref = torch.empty(B, H, N, 64, device=dev)
    for b in range(B):
        for h in range(H):
            s = (q[b, h] @ k[b, h].t()) * math.log(2.0)   # the kernel's scores are in log2 units
            ref[b, h] = torch.softmax(s, dim=-1) @ v[b, h]
    ref = ref.permute(0, 2, 1, 3).reshape(B * N, D)
    got = out.float()
    err = (got - ref).abs().max().item()
    scale = ref.abs().max().item()
    tol = 2.5e-2 * scale
    bad = ((got - ref).abs() > tol).nonzero()
    first_bad = bad[0].tolist() if bad.numel() else None
    return _report(name, rc == 0 and err <= tol and bool(torch.isfinite(got).all()) and was_redone == redone, rc=rc, max_abs_err=err,
                   ref_absmax=scale, tol=tol, n_bad=int(bad.shape[0]), first_bad=first_bad, redone=was_redone)


def check_mlp(name, M, pair=0):
    """Fused fc1 -> GELU(erf) -> fc2 -> +x kernel (A = LayerNorm(x) in bf16) vs fp32 torch (bf16 operand rounding emulated for the
    reference's inputs only through the tolerance: 1 % of the output's max-abs)."""
    torch, L, lib = _imports()
    torch.manual_seed(7)
    dev = "cuda"
    x = torch.randn(M, 384, device=dev) * 1.5 + 0.2
    g = 1.0 + 0.1 * torch.randn(384, device=dev)
    b = 0.1 * torch.randn(384, device=dev)
    W1 = (torch.randn(1536, 384, device=dev) * 0.05).to(torch.bfloat16)
    b1 = 0.1 * torch.randn(1536, device=dev)
    W2 = (torch.randn(384, 1536, device=dev) * 0.03).to(torch.bfloat16)
    b2 = 0.1 * torch.randn(384, device=dev)
    F = torch.nn.functional
    ln = F.layer_norm(x, (384,), g, b, 1e-6)
    hid = F.gelu(F.linear(ln.to(torch.bfloat16).float(), W1.float(), b1))
    ref = x + F.linear(hid.to(torch.bfloat16).float(), W2.float(), b2)
    y = x.clone()
    A = ln.to(torch.bfloat16).contiguous()
    rc = lib.dinoseg_op_mlp_ex(_ptr(y), _ptr(A), _ptr(W1), _ptr(b1), _ptr(W2), _ptr(b2), M, pair, None)
    torch.cuda.synchronize()
    err = (y - ref).abs().max().item()
    scale = ref.abs().max().item()
    tol = 1e-2 * scale
    bad = ((y - ref).abs() > tol).nonzero()
    return _report(name, rc == 0 and err <= tol and bool(torch.isfinite(y).all()), rc=rc, max_abs_err=err,
                   ref_absmax=scale, tol=tol, n_bad=int(bad.shape[0]), first_bad=bad[0].tolist() if bad.numel() else None)


def check_mlp_ln(name, M, pair=0):
    """The fused MLP kernel normalising the residual stream itself, with LayerNorm2's gamma / beta folded into fc1
    (dinoseg_op_fold_ln + dinoseg_op_mlp_ln), against fp32 torch and against the two-kernel path (LayerNorm kernel, then the
    MLP kernel on its bf16 output): same function, operands rounded to bf16 at different points."""
    torch, L, lib = _imports()
    torch.manual_seed(8)
    dev = "cuda"
    x = torch.randn(M, 384, device=dev) * 1.5 + 0.2
    x[3] *= 40.0                                   # a row with a large mean / spread
    g = 1.0 + 0.1 * torch.randn(384, device=dev)
    b = 0.1 * torch.randn(384, device=dev)
    W1 = torch.randn(1536, 384, device=dev) * 0.05
    b1 = 0.1 * torch.randn(1536, device=dev)
    W2 = (torch.randn(384, 1536, device=dev) * 0.03).to(torch.bfloat16)
    b2 = 0.1 * torch.randn(384, device=dev)
    F = torch.nn.functional
    ref = x + F.linear(F.gelu(F.linear(F.layer_norm(x, (384,), g, b, 1e-6), W1, b1)), W2.float(), b2)     # fp32 throughout
    A = torch.zeros(M, 384, device=dev, dtype=torch.bfloat16)
    rc0 = lib.dinoseg_op_layernorm(_ptr(x), _ptr(g), _ptr(b), _ptr(A), M, 384, 1e-6, None)
    two = x.clone()
    W1b = W1.to(torch.bfloat16)
    rc1 = lib.dinoseg_op_mlp_ex(_ptr(two), _ptr(A), _ptr(W1b), _ptr(b1), _ptr(W2), _ptr(b2), M, pair, None)
    W1f = torch.zeros(1536, 384, device=dev, dtype=torch.bfloat16)
    b1f = torch.zeros(1536, device=dev)
    rc2 = lib.dinoseg_op_fold_ln(_ptr(W1), _ptr(b1), _ptr(g), _ptr(b), 1536, 384, _ptr(W1f), _ptr(b1f), None)
    one = x.clone()
    rc3 = lib.dinoseg_op_mlp_ln(_ptr(one), 1e-6, _ptr(W1f), _ptr(b1f), _ptr(W2), _ptr(b2), M, pair, None)
    torch.cuda.synchronize()
    fold_ok = bool(torch.equal(W1f, (W1 * g).to(torch.bfloat16))) and (b1f - (b1 + W1 @ b)).abs().max().item() <= 1e-5
    scale = (ref - x).abs().max().item()           # size of the MLP update (x itself is added exactly)
    err1, err2 = (one - ref).abs().max().item(), (two - ref).abs().max().item()
    ok = rc0 == 0 and rc1 == 0 and rc2 == 0 and rc3 == 0 and fold_ok and err1 <= 1e-2 * scale and err2 <= 1e-2 * scale \
        and bool(torch.isfinite(one).all())
    return _report(name, ok, rc=[rc0, rc1, rc2, rc3], fold_exact=fold_ok, max_abs_err_fused=err1, max_abs_err_two_kernels=err2,
                   update_absmax=scale, max_diff_fused_vs_two_kernels=(one - two).abs().max().item())


def check_layernorm(name, M, D):
    torch, L, lib = _imports()
    torch.manual_seed(3)
    x = torch.randn(M, D, device="cuda") * 2 + 0.3
    g = torch.randn(D, device="cuda") * 0.1 + 1
    b = torch.randn(D, device="cuda") * 0.1
    y = torch.zeros(M, D, device="cuda", dtype=torch.bfloat16)
    rc = lib.dinoseg_op_layernorm(_ptr(x), _ptr(g), _ptr(b), _ptr(y), M, D, 1e-6, None)
    torch.cuda.synchronize()
    ref = torch.nn.functional.layer_norm(x, (D,), g, b, 1e-6)
    err = (y.float() - ref.to(torch.bfloat16).float()).abs().max().item()
    # identical up to one bf16 ulp of the largest value
    return _report(name, rc == 0 and err <= 0.04, rc=rc, max_abs_err=err)


def check_posembed(name, g, D=384, G0=28):
    torch, L, lib = _imports()
    torch.manual_seed(4)
    pos = torch.randn(1, G0 * G0 + 1, D, device="cuda")
    out = torch.zeros(g * g + 1, D, device="cuda")
    rc = lib.dinoseg_op_posembed(_ptr(pos), _ptr(out), G0, g, D, None)
    torch.cuda.synchronize()
    # reference semantics: vision_transformer.py:202-222 evaluated by torch on the CPU
    pc = pos.cpu()
    if g == G0:
        ref = pc[0]
    else:
        patch = pc[:, 1:].reshape(1, G0, G0, D).permute(0, 3, 1, 2)
        sf = (g + 0.1) / math.sqrt(G0 * G0)
        patch = torch.nn.functional.interpolate(patch, scale_factor=(sf, sf), mode="bicubic")
        assert patch.shape[-1] == g and patch.shape[-2] == g
        ref = torch.cat((pc[:, 0], patch.permute(0, 2, 3, 1).reshape(-1, D)), dim=0)
    err = (out.cpu() - ref).abs().max().item()
    return _report(name, rc == 0 and err <= 2e-5, rc=rc, max_abs_err=err)


def check_im2col(name, B, g):
    """im2col emits the bf16x3 operand [hi | lo] of the patch-embed GEMM (2 x 192 columns)."""
    torch, L, lib = _imports()
    torch.manual_seed(5)
    r = g * 8
    frames = torch.randn(B, 3, r, r, device="cuda")
    A = torch.zeros(B * g * g, 384, device="cuda", dtype=torch.bfloat16)
    rc = lib.dinoseg_op_im2col(_ptr(frames), _ptr(A), B, g, None)
    torch.cuda.synchronize()
    ref = torch.nn.functional.unfold(frames, kernel_size=8, stride=8)  # [B, 192, P], k = c*64+ky*8+kx
    ref = ref.transpose(1, 2).reshape(B * g * g, 192)
    hi = ref.to(torch.bfloat16)
    lo = (ref - hi.float()).to(torch.bfloat16)
    same = bool((A[:, :192] == hi).all()) and bool((A[:, 192:] == lo).all())
    return _report(name, rc == 0 and same, rc=rc, identical=same)


def check_argmax_replicate(name, B, g, C, p):
    torch, L, lib = _imports()
    import numpy as np
    torch.manual_seed(6)
    lp = torch.randn(B * g * g, C, device="cuda")
    # ties and NaNs: torch.argmax -> first max wins, NaN counts as max
    lp[5] = 0.25
    lp[7, 2] = lp[7, 4] = 9.0
    lp[9, 3] = float("nan")
    lp[11, 1] = float("nan"); lp[11, 5] = float("nan")
    lp[13] = float("-inf")
    low = torch.zeros(B, g, g, device="cuda", dtype=torch.uint8)
    lab = torch.zeros(B, g * p, g * p, device="cuda", dtype=torch.int64)
    rc = lib.dinoseg_argmax_replicate(_ptr(lp), B, g, C, p, _ptr(low), _ptr(lab), None)
    torch.cuda.synchronize()
    ref_low = torch.argmax(lp.cpu(), dim=-1).numpy().reshape(B, g, g)
    ref = np.stack([np.kron(ref_low[b], np.ones((p, p), dtype=int)) for b in range(B)])
    ok = bool((low.cpu().numpy() == ref_low).all()) and bool((lab.cpu().numpy() == ref).all())
    return _report(name, rc == 0 and ok, rc=rc, identical=ok)


def _checks():
    from dino_b200 import _lib as L
    return {
        "layernorm_384": lambda: check_layernorm("layernorm_384", 1000, 384),
        "layernorm_768": lambda: check_layernorm("layernorm_768", 333, 768),
        "posembed_30": lambda: check_posembed("posembed_30", 30),
        "posembed_60": lambda: check_posembed("posembed_60", 60),
        "posembed_28": lambda: check_posembed("posembed_28", 28),
        "posembed_vitb_60": lambda: check_posembed("posembed_vitb_60", 60, D=768),
        "im2col": lambda: check_im2col("im2col", 2, 30),
        "argmax_replicate": lambda: check_argmax_replicate("argmax_replicate", 2, 30, 7, 16),
        "argmax_replicate_odd": lambda: check_argmax_replicate("argmax_replicate_odd", 1, 9, 7, 53),
        "gemm_tile": lambda: check_gemm("gemm_tile", 128, 128, 64, L.EPI_RELU_F32, with_bias=False),
        "gemm_k384": lambda: check_gemm("gemm_k384", 128, 128, 384, L.EPI_RELU_F32),
        "gemm_qkv": lambda: check_gemm("gemm_qkv", 1000, 1152, 384, L.EPI_BF16),
        "gemm_pair_small": lambda: check_gemm_pair("gemm_pair_small", 128, 192, 64),
        "gemm_pair_qkv": lambda: check_gemm_pair("gemm_pair_qkv", 1000, 1152, 384),
        "gemm_pair_big": lambda: check_gemm_pair("gemm_pair_big", 148 * 128 * 3 + 300, 1152, 384),
        "gemm_pair_vitb": lambda: check_gemm_pair("gemm_pair_vitb", 901 * 3, 2304, 768),
        "gemm_pair_gelu": lambda: check_gemm_pair("gemm_pair_gelu", 901 * 3, 3072, 768, L.EPI_GELU_BF16),
        "gemm_pair_resid": lambda: check_gemm_pair("gemm_pair_resid", 901 * 3, 768, 3072, L.EPI_RESID_F32),
        "gemm_gelu": lambda: check_gemm("gemm_gelu", 901, 1536, 384, L.EPI_GELU_BF16),
        "gemm_resid_k1536": lambda: check_gemm("gemm_resid_k1536", 901, 384, 1536, L.EPI_RESID_F32),
        "gemm_patch": lambda: check_gemm("gemm_patch", 2 * 900, 384, 192, L.EPI_PATCH_F32, P=900, Ntok=901),
        "gemm_head": lambda: check_gemm("gemm_head", 901, 200, 384, L.EPI_RELU_F32),
        "gemm_big": lambda: check_gemm("gemm_big", 8 * 3601, 1152, 384, L.EPI_BF16),
        "attn_1tile": lambda: check_attention("attn_1tile", 1, 128, 1),
        "attn_ragged_small": lambda: check_attention("attn_ragged_small", 1, 100, 2),
        "attn_2tiles": lambda: check_attention("attn_2tiles", 1, 256, 1),
        "attn_901": lambda: check_attention("attn_901", 2, 901, 6),
        "attn_3601": lambda: check_attention("attn_3601", 1, 3601, 6),
        "attn_vitb_901": lambda: check_attention("attn_vitb_901", 1, 901, 12),
        # scores beyond +-100 log2 units: the kernel without row maxima flags the launch and the classic kernel redoes it
        "attn_wide_901": lambda: check_attention("attn_wide_901", 2, 901, 6, spread=16.0, redone=1),
        "attn_shifted_901": lambda: check_attention("attn_shifted_901", 2, 901, 6, spread=4.0, shift=6.0, redone=1),
        # logits up to about +-60: large, but still inside the range of the kernel without row maxima
        "attn_spread8_901": lambda: check_attention("attn_spread8_901", 2, 901, 6, spread=8.0),
        "mlp_1block": lambda: check_mlp("mlp_1block", 128),
        "mlp_ragged": lambda: check_mlp("mlp_ragged", 901),
        "mlp_multi": lambda: check_mlp("mlp_multi", 148 * 128 * 2 + 77),
        "mlp_pair_1block": lambda: check_mlp("mlp_pair_1block", 128, 1),
        "mlp_pair_ragged": lambda: check_mlp("mlp_pair_ragged", 901, 1),
        "mlp_pair_multi": lambda: check_mlp("mlp_pair_multi", 148 * 128 * 2 + 77, 1),
        "mlp_ln_ragged": lambda: check_mlp_ln("mlp_ln_ragged", 901),
        "mlp_ln_multi": lambda: check_mlp_ln("mlp_ln_multi", 148 * 128 * 2 + 77),
        "mlp_ln_pair_ragged": lambda: check_mlp_ln("mlp_ln_pair_ragged", 901, 1),
        "mlp_ln_pair_multi": lambda: check_mlp_ln("mlp_ln_pair_multi", 148 * 128 * 3 + 300, 1),
    }


def check_names():
    return [
        "layernorm_384", "layernorm_768", "posembed_30", "posembed_60", "posembed_28", "posembed_vitb_60", "im2col",
        "argmax_replicate", "argmax_replicate_odd", "gemm_tile", "gemm_k384", "gemm_qkv", "gemm_pair_small", "gemm_pair_qkv", "gemm_pair_big", "gemm_pair_vitb", "gemm_pair_gelu", "gemm_pair_resid", "gemm_gelu",
        "gemm_resid_k1536", "gemm_patch", "gemm_head", "gemm_big", "attn_1tile", "attn_ragged_small", "attn_2tiles",
        "attn_901", "attn_3601", "attn_vitb_901", "mlp_1block", "mlp_ragged", "mlp_multi", "mlp_pair_1block", "mlp_pair_ragged", "mlp_pair_multi",
        "mlp_ln_ragged", "mlp_ln_multi", "mlp_ln_pair_ragged", "mlp_ln_pair_multi",
    ]


def run_check(name):
    return _checks()[name]()


def main():
    if len(sys.argv) > 1 and sys.argv[1] != "--all":
        ok = _checks()[sys.argv[1]]()
        sys.exit(0 if ok else 1)
    names = list(_checks().keys())
    results = {}
    for n in names:
        t0 = time.time()
        try:
            proc = subprocess.run([sys.executable, os.path.abspath(__file__), n], capture_output=True, text=True,
                                  timeout=180)
            out = proc.stdout + proc.stderr
            line = [l for l in out.splitlines() if l.startswith("CHECK ")]
            results[n] = (proc.returncode == 0, line[-1] if line else out[-1500:])
        except subprocess.TimeoutExpired:
            results[n] = (False, "TIMEOUT")
        print(f"[{'PASS' if results[n][0] else 'FAIL'}] {n} ({time.time() - t0:.1f}s) {results[n][1]}", flush=True)
    nfail = sum(1 for ok, _ in results.values() if not ok)
    print(f"SUMMARY {len(names) - nfail}/{len(names)} passed")
    sys.exit(1 if nfail else 0)


if __name__ == "__main__":
    main()

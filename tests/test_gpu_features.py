"""Backbone features on a real B200: model.dino(x), model.dino.get_intermediate_layers(x, n) and DINOSeg.features
(dinoseg_features / dinoseg_features_u8, one pass over the blocks, no head) against the unmodified reference
(tests/golden norm_rows) and the CPU reference (tests/features_ref.py).

Tolerances (features_ref.py): bf16 GEMM / attention operands, fp32 residual stream and final LayerNorm -
max-abs error <= 1e-2 (reference_init) / 4e-2 (trained_like stress weights) of max |ref|, Frobenius error <= 2.5e-2
of the Frobenius norm, every token's cosine similarity >= 0.999.  Measured values are appended to the parity
statistics of the end-to-end tests (test_gpu_e2e._record).
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN_CASES, load_golden
from dino_b200 import DINOSeg, _lib, synthetic
from features_ref import FRO_REL, MAX_REL, MIN_COS, feature_errors, intermediate_layers
from oracle import dinoseg_oracle as O
from test_gpu_e2e import _record

pytestmark = pytest.mark.gpu


def _model(arch, n_blocks, seed, variant, n_classes=7, head="mlp"):
    cfg = synthetic.make_config(arch, n_blocks, n_classes, head=head)
    sd = synthetic.init_state_dict(cfg, seed, variant)
    m = DINOSeg(head=head, n_blocks=n_blocks, n_classes=n_classes, arch=arch)
    m.load_state_dict(sd, strict=True)
    return m.to("cuda:0"), cfg, sd


def _check(tag, got, ref, variant):
    rel, fro, cos = feature_errors(got, ref)
    _record(case=tag, features_max_rel=rel, features_fro_rel=fro, features_min_cos=cos, variant=variant)
    assert rel <= MAX_REL[variant] and fro <= FRO_REL and cos >= MIN_COS, (tag, rel, fro, cos)


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_dino_forward_against_reference_golden(name):
    """model.dino(x) at the rows the reference stored (oracle/make_golden.py: norm_rows = m.dino(x)[:, rows])."""
    gd = load_golden(name)
    meta = gd["meta"]
    m, cfg, sd = _model(meta["arch"], meta["n_blocks"], meta["seed"], meta["variant"], meta["n_classes"],
                        meta.get("head", "mlp"))
    x = synthetic.make_frames(meta["batch"], meta["res"], meta["seed"])
    f = m.dino(x.cuda())
    torch.cuda.synchronize()
    n = (meta["res"] // 8) ** 2 + 1
    assert tuple(f.shape) == (meta["batch"], n, cfg["embed_dim"]) and f.dtype == torch.float32
    assert torch.isfinite(f).all()
    _check(name, f[:, gd["rows"]].cpu(), torch.from_numpy(gd["norm_rows"]), meta["variant"])


@pytest.mark.parametrize("res,nb,batch", [(64, 1, 5), (224, 2, 1), (496, 1, 1), (8, 1, 3), (960, 1, 1)])
def test_dino_forward_against_oracle_edge_resolutions(res, nb, batch):
    """Whole feature tensors at the ragged / extreme sizes of the segmentation tests: one 128-key tile, the identity
    positional table, 496 px, one patch per frame, 14401 tokens."""
    m, cfg, sd = _model("vit_small", nb, 11, "reference_init")
    x = synthetic.make_frames(batch, res, seed=res)
    f = m.dino(x.cuda())
    torch.cuda.synchronize()
    torch.set_num_threads(os.cpu_count() or 1)
    ref = O.backbone(sd, cfg, x)
    assert f.shape == ref.shape
    _check(f"features_oracle_{res}", f.cpu(), ref, "reference_init")


@pytest.mark.parametrize("arch,nb,variant,res,batch", [("vit_small", 3, "trained_like", 240, 2),
                                                       ("vit_base", 4, "reference_init", 240, 1)])
def test_get_intermediate_layers(arch, nb, variant, res, batch):
    """n = 1 .. n_blocks and n > n_blocks: min(n, n_blocks) layers, oldest first, each within the bars of the CPU
    reference; the last one is model.dino(x) bit for bit, and the k-th from last does not depend on n."""
    m, cfg, sd = _model(arch, nb, 5, variant)
    x = synthetic.make_frames(batch, res, seed=6)
    xd = x.cuda()
    full = m.dino(xd)
    got = {n: m.dino.get_intermediate_layers(xd, n=n) for n in range(1, nb + 3)}
    torch.cuda.synchronize()
    ref = intermediate_layers(sd, cfg, x, nb)
    for n, layers in got.items():
        assert isinstance(layers, list) and len(layers) == min(n, nb), n
        assert torch.equal(layers[-1], full), n
        for k in range(1, len(layers) + 1):
            assert torch.equal(layers[-k], got[nb][-k]), (n, k)
    for i, layer in enumerate(got[nb]):
        _check(f"intermediate_{arch}_{variant}_block{i}", layer.cpu(), ref[i], variant)


def test_full_size_batch_properties():
    """Bench shape (ViT-S/8, 3 blocks, 480 px, batch 64): deterministic, frame-independent, the same with the single-CTA
    kernels as with the CTA pairs, and normalised tokens under the reference-init norm (gamma = 1, beta = 0)."""
    lib = _lib.load()
    m, cfg, sd = _model("vit_small", 3, 0, "reference_init")
    assert torch.equal(sd["dino.norm.weight"], torch.ones(384)) and torch.equal(sd["dino.norm.bias"], torch.zeros(384))
    x = synthetic.make_frames(64, 480, seed=1).cuda()
    f = m.dino(x)
    f2 = m.dino(x)
    torch.cuda.synchronize()
    assert tuple(f.shape) == (64, 3601, 384) and torch.isfinite(f).all()
    assert torch.equal(f, f2)
    for sl in (slice(0, 1), slice(5, 8), slice(61, 64)):
        fs = m.dino(x[sl].contiguous())
        torch.cuda.synchronize()
        assert torch.equal(fs, f[sl]), sl
    assert lib.dinoseg_set_pair_kernels(m._handle, 0) == 0
    try:
        single = m.dino(x)
        torch.cuda.synchronize()
    finally:
        assert lib.dinoseg_set_pair_kernels(m._handle, 1) == 0
    assert torch.equal(single, f)
    fd = f.double()
    mean = fd.mean(-1)
    var = fd.var(-1, unbiased=False)
    _record(case="features_full_size_b64_480", token_mean_absmax=float(mean.abs().max()),
            token_var_dev_max=float((var - 1).abs().max()))
    assert float(mean.abs().max()) <= 1e-5 and float((var - 1).abs().max()) <= 1e-3


@pytest.mark.parametrize("arch,nb,variant,head", [("vit_small", 2, "reference_init", "mlp"), ("vit_small", 2, "trained_like", "mlp"),
                                                  ("vit_small", 1, "reference_init", "linear"), ("vit_base", 1, "trained_like", "mlp")])
def test_features_feed_the_head_like_the_segmentation_path(arch, nb, variant, head):
    """The fp32 head of the CPU reference on the GPU features reproduces the log-probs of model(x): both start from the
    same residual stream, and the head evaluates its own LayerNorm and Linear layers in bf16x3."""
    m, cfg, sd = _model(arch, nb, 8, variant, head=head)
    x = synthetic.make_frames(2, 240, seed=3).cuda()
    f = m.dino(x)
    lp = m(x)
    torch.cuda.synchronize()
    d = cfg["embed_dim"]
    ref = O.head(sd, f[:, 1:].reshape(-1, d).cpu())
    rng = float(ref.max() - ref.min())
    err = float((lp.cpu() - ref).abs().max())
    _record(case=f"features_head_{arch}_{variant}_{head}", max_abs=err, range=rng)
    assert err <= 2e-4 * max(1.0, rng), (err, rng)


@pytest.mark.parametrize("arch,head_launches", [("vit_small", 1), ("vit_base", 4)])
def test_features_leave_the_segmentation_path_alone(arch, head_launches):
    """A features call on the same handle changes neither the outputs nor the launches of the next forward; the feature
    pass is the forward without its head kernels (ViT-S: the fused head; ViT-B: LayerNorm, two GEMMs, tail) plus one
    fp32 LayerNorm per requested block."""
    nb = 3 if arch == "vit_small" else 2
    m, cfg, sd = _model(arch, nb, 4, "trained_like")
    x = synthetic.make_frames(3, 240, seed=2).cuda()
    lp0, low0, lab0 = m.infer(x, want_logprobs=True, want_lowres=True, want_labels=True)
    n_fwd = m.last_launch_count()
    for n in range(1, nb + 2):
        m.features(x, n)
        assert m.last_launch_count() == n_fwd - head_launches + min(n, nb), n
    lp1, low1, lab1 = m.infer(x, want_logprobs=True, want_lowres=True, want_labels=True)
    torch.cuda.synchronize()
    assert m.last_launch_count() == n_fwd
    assert torch.equal(lp0, lp1) and torch.equal(low0, low1) and torch.equal(lab0, lab1)


@pytest.mark.parametrize("hw,res", [((480, 640), 240), ((360, 500), 480), ((480, 480), 480)])
def test_raw_frame_features_are_bit_exact(hw, res):
    """uint8 HWC frames through the fused resize / normalise im2col give the features of the preprocessing oracle's fp32
    frames, bit for bit."""
    from oracle import preproc_oracle as P
    m, cfg, sd = _model("vit_small", 2, 2, "trained_like")
    rng = np.random.default_rng(res + hw[1])
    imgs = rng.integers(0, 256, (3, hw[0], hw[1], 3), dtype=np.uint8)
    f_u8 = m.features(torch.from_numpy(imgs).cuda(), n=2, resolution=res)
    x = torch.from_numpy(np.stack([P.preprocess(im, res) for im in imgs])).cuda()
    f = m.features(x, n=2)
    torch.cuda.synchronize()
    assert tuple(f.shape) == (2, 3, (res // 8) ** 2 + 1, 384)
    assert torch.equal(f_u8, f)


@pytest.mark.parametrize("M,D", [(1000, 384), (333, 768), (1, 384), (37, 768), (148 * 32 + 5, 384)])
def test_layernorm_f32_kernel(M, D):
    """dinoseg_op_layernorm_f32 against fp64 torch (fp32 rounding only), rows beyond M untouched, and the same values
    as the bf16 LayerNorm of the forward before its rounding to bf16."""
    lib = _lib.load()
    torch.manual_seed(M + D)
    x = torch.randn(M, D, device="cuda") * 2 + 0.3
    g = torch.randn(D, device="cuda") * 0.1 + 1
    b = torch.randn(D, device="cuda") * 0.1
    y = torch.full((M + 1, D), 7.0, device="cuda")
    yb = torch.zeros(M, D, device="cuda", dtype=torch.bfloat16)
    assert lib.dinoseg_op_layernorm_f32(x.data_ptr(), g.data_ptr(), b.data_ptr(), y.data_ptr(), M, D, 1e-6, None) == 0
    assert lib.dinoseg_op_layernorm(x.data_ptr(), g.data_ptr(), b.data_ptr(), yb.data_ptr(), M, D, 1e-6, None) == 0
    torch.cuda.synchronize()
    ref = torch.nn.functional.layer_norm(x.double(), (D,), g.double(), b.double(), 1e-6)
    err = float((y[:M].double() - ref).abs().max() / ref.abs().max())
    _record(case=f"layernorm_f32_{M}_{D}", max_rel=err)
    assert err <= 2e-6, err
    assert (y[M] == 7.0).all()
    assert torch.equal(y[:M].to(torch.bfloat16), yb)
    assert lib.dinoseg_op_layernorm_f32(x.data_ptr(), g.data_ptr(), b.data_ptr(), y.data_ptr(), M, 512, 1e-6, None) != 0


def test_c_abi_misuse_is_reported():
    """Bad n_last, NULL out, no resolution, too small a workspace: an error code and a message, never a crash."""
    lib = _lib.load()
    h = C.c_void_p()
    cfg = _lib.DinosegCfg(384, 6, 1536, 1, 8, 28, 7, 200, 100, 0, 1e-6)
    assert lib.dinoseg_create(C.byref(cfg), 0, C.byref(h)) == 0
    x = torch.zeros(1, 3, 64, 64, device="cuda")
    out = torch.zeros(1, 1, 65, 384, device="cuda")
    ws = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
    try:
        assert lib.dinoseg_features(h, x.data_ptr(), 1, 1, out.data_ptr(), ws.data_ptr(), ws.numel(), None) != 0
        assert "set_resolution" in _lib.last_error(h)
    finally:
        lib.dinoseg_destroy(h)
    m, _, _ = _model("vit_small", 2, 1, "reference_init")
    m.features(x)                                          # handle, resolution 64 and workspace in place
    ws = m._workspace
    hd = m._handle
    assert lib.dinoseg_features(hd, x.data_ptr(), 1, 0, out.data_ptr(), ws.data_ptr(), ws.numel(), None) != 0
    assert "n_last" in _lib.last_error(hd)
    assert lib.dinoseg_features(hd, x.data_ptr(), 1, 1, None, ws.data_ptr(), ws.numel(), None) != 0
    assert "out" in _lib.last_error(hd)
    assert lib.dinoseg_features(hd, x.data_ptr(), 1, 1, out.data_ptr(), ws.data_ptr(), 1024, None) != 0
    assert "workspace too small" in _lib.last_error(hd)
    u8 = torch.zeros(1, 64, 64, 3, dtype=torch.uint8, device="cuda")
    mean, std = (C.c_float * 3)(0.5, 0.5, 0.5), (C.c_float * 3)(0.25, 0.25, 0.25)
    assert lib.dinoseg_features_u8(hd, u8.data_ptr(), 1, 64, 64, mean, std, -1, out.data_ptr(), ws.data_ptr(), ws.numel(),
                                   None) != 0
    assert lib.dinoseg_features_u8(hd, u8.data_ptr(), 1, 0, 64, mean, std, 1, out.data_ptr(), ws.data_ptr(), ws.numel(),
                                   None) != 0
    assert lib.dinoseg_features(hd, x.data_ptr(), 1, 1, out.data_ptr(), ws.data_ptr(), ws.numel(), None) == 0
    torch.cuda.synchronize()
    assert torch.equal(out[0], m.dino(x))
    with pytest.raises(ValueError):
        m.dino(torch.zeros(1, 3, 64, 48, device="cuda"))       # not square
    with pytest.raises(ValueError):
        m.dino(torch.zeros(1, 3, 60, 60, device="cuda"))       # not a multiple of 8
    with pytest.raises(ValueError):
        m.dino.get_intermediate_layers(x, n=0)

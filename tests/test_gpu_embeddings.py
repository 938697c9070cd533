"""Image embeddings on a real B200: DINOSeg.embeddings (dinoseg_embeddings / dinoseg_embeddings_u8) against the
unmodified reference (tests/golden norm_rows[:, 0]), the CPU reference (tests/embeddings_ref.py) and the GPU's own
features().

Bars are the feature bars of features_ref (MAX_REL, FRO_REL, MIN_COS): the CLS-only tail rounds the attention output,
the proj / MLP operands and V to bf16 as the full-size path does.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import embeddings_ref as E
import rect_ref
from conftest import GOLDEN_CASES, load_golden
from dino_b200 import DINOSeg, _lib, synthetic
from features_ref import FRO_REL, MAX_REL, MIN_COS, feature_errors
from test_gpu_e2e import _record

pytestmark = pytest.mark.gpu


def _model(arch, n_blocks, seed, variant, n_classes=7, head="mlp", sd=None):
    cfg = synthetic.make_config(arch, n_blocks, n_classes, head=head)
    if sd is None:
        sd = synthetic.init_state_dict(cfg, seed, variant)
    m = DINOSeg(head=head, n_blocks=n_blocks, n_classes=n_classes, arch=arch)
    m.load_state_dict(sd, strict=True)
    return m.to("cuda:0"), cfg, sd


def _frames(batch, hw, seed):
    if hw[0] == hw[1]:
        return synthetic.make_frames(batch, hw[0], seed)
    g = torch.Generator().manual_seed(seed)
    return torch.randn(batch, 3, hw[0], hw[1], generator=g)


def _check(tag, got, ref, variant):
    assert torch.isfinite(got).all(), tag
    rel, fro, cos = feature_errors(got.cpu(), ref)
    _record(case=tag, emb_max_rel=rel, emb_fro_rel=fro, emb_min_cos=cos, variant=variant)
    assert rel <= MAX_REL[variant] and fro <= FRO_REL and cos >= MIN_COS, (tag, rel, fro, cos)


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_cls_embedding_against_reference_golden(name):
    """embeddings(x, 1) is the reference's CLS embedding: norm_rows[:, 0] (rows[0] == 0) of model.dino(x)."""
    gd = load_golden(name)
    meta = gd["meta"]
    assert int(gd["rows"][0]) == 0
    m, cfg, sd = _model(meta["arch"], meta["n_blocks"], meta["seed"], meta["variant"], meta["n_classes"],
                        meta.get("head", "mlp"))
    x = synthetic.make_frames(meta["batch"], meta["res"], meta["seed"])
    e = m.embeddings(x.cuda())
    torch.cuda.synchronize()
    assert tuple(e.shape) == (meta["batch"], cfg["embed_dim"]) and e.dtype == torch.float32
    _check(f"emb_golden_{name}", e, torch.from_numpy(gd["norm_rows"][:, 0]), meta["variant"])


@pytest.mark.parametrize("arch,nb,variant,hw,batch", [
    ("vit_small", 3, "trained_like", (224, 224), 2),
    ("vit_small", 2, "reference_init", (64, 64), 5),
    ("vit_small", 3, "reference_init", (480, 480), 1),
    ("vit_small", 2, "trained_like", (480, 640), 2),
    ("vit_base", 2, "trained_like", (64, 64), 3),
    ("vit_base", 2, "reference_init", (224, 224), 1),
    ("vit_base", 4, "reference_init", (480, 480), 4),
])
def test_embeddings_against_cpu_reference(arch, nb, variant, hw, batch):
    """Every n in 1 .. n_blocks + 1 and avgpool on / off against upstream's expressions on the CPU reference layers."""
    m, cfg, sd = _model(arch, nb, 7, variant)
    x = _frames(batch, hw, seed=hw[1] + batch)
    layers = E.intermediate_layers(sd, cfg, x, nb)
    xd = x.cuda()
    d = cfg["embed_dim"]
    for n in range(1, nb + 2):
        e = m.embeddings(xd, n)
        n_out = min(n, nb)
        assert tuple(e.shape) == (batch, n_out * d), n
        _check(f"emb_{arch}_{variant}_{hw[0]}x{hw[1]}_b{batch}_n{n}", e, E.from_layers(layers[nb - n_out:]), variant)
    e = m.embeddings(xd, 1, avgpool=True)
    assert tuple(e.shape) == (batch, 2 * d)
    _check(f"emb_avgpool_{arch}_{variant}_{hw[0]}x{hw[1]}_b{batch}", e, E.from_layers(layers[-1:], avgpool=True), variant)


@pytest.mark.parametrize("arch,nb,hw,batch", [("vit_small", 3, (480, 480), 4), ("vit_base", 4, (240, 240), 3),
                                              ("vit_small", 2, (480, 640), 2)])
def test_consistency_with_features(arch, nb, hw, batch):
    """Earlier blocks' CLS slices and the whole avgpool CLS output are features()' CLS rows bit for bit; the CLS-only last
    slice lies within the feature bars of features()' last CLS row; the patch mean is within 1e-5 of features()'."""
    m, cfg, sd = _model(arch, nb, 3, "trained_like")
    x = _frames(batch, hw, seed=9).cuda()
    d = cfg["embed_dim"]
    for n in range(1, nb + 1):
        f = m.features(x, n)[:, :, 0]                              # [n, B, D]
        e = m.embeddings(x, n).reshape(batch, n, d).permute(1, 0, 2)
        torch.cuda.synchronize()
        assert torch.equal(e[:-1], f[:-1]), n
        _check(f"emb_vs_features_{arch}_{hw[0]}x{hw[1]}_n{n}", e[-1], f[-1].cpu(), "trained_like")
    f1 = m.features(x, 1)[0]
    pooled = m.embeddings(x, 1, avgpool=True)
    torch.cuda.synchronize()
    assert torch.equal(pooled[:, 0::2], f1[:, 0])
    ref = f1[:, 1:].double().mean(1)
    err = float((pooled[:, 1::2].double() - ref).abs().max() / ref.abs().max())
    _record(case=f"emb_patch_mean_{arch}_{hw[0]}x{hw[1]}", max_rel=err)
    assert err <= 1e-5, err


def test_determinism_and_frame_independence():
    """Bench shape (ViT-S/8, 3 blocks, 480 px, batch 64) and a 130-frame batch at 64 px (two row blocks of the M = B
    GEMMs, the second one partial): two calls are bit-identical, every sub-batch (B = 1 included) equals its rows of
    the full batch, and the single-CTA kernels give the CTA pairs' bits."""
    lib = _lib.load()
    m, cfg, sd = _model("vit_small", 3, 0, "reference_init")
    for res, batch, slices in ((480, 64, (slice(0, 1), slice(5, 8), slice(63, 64))),
                               (64, 130, (slice(0, 1), slice(127, 130), slice(0, 129)))):
        x = synthetic.make_frames(batch, res, seed=1).cuda()
        for kw in ({"n": 1}, {"n": 3}, {"n": 1, "avgpool": True}):
            e = m.embeddings(x, **kw)
            e2 = m.embeddings(x, **kw)
            torch.cuda.synchronize()
            assert torch.isfinite(e).all() and torch.equal(e, e2), (res, kw)
            for sl in slices:
                es = m.embeddings(x[sl].contiguous(), **kw)
                torch.cuda.synchronize()
                assert torch.equal(es, e[sl]), (res, kw, sl)
            assert lib.dinoseg_set_pair_kernels(m._handle, 0) == 0
            try:
                single = m.embeddings(x, **kw)
                torch.cuda.synchronize()
            finally:
                assert lib.dinoseg_set_pair_kernels(m._handle, 1) == 0
            assert torch.equal(single, e), (res, kw)


def test_vit_b_single_frame_pairs_and_single_cta():
    """ViT-B at B = 1: fc1 / fc2 as CTA pairs with one row block give the single-CTA kernels' bits."""
    lib = _lib.load()
    m, cfg, sd = _model("vit_base", 2, 4, "trained_like")
    x = synthetic.make_frames(1, 224, seed=4).cuda()
    e = m.embeddings(x, 2)
    assert lib.dinoseg_set_pair_kernels(m._handle, 0) == 0
    try:
        single = m.embeddings(x, 2)
        torch.cuda.synchronize()
    finally:
        assert lib.dinoseg_set_pair_kernels(m._handle, 1) == 0
    assert torch.equal(single, e)


@pytest.mark.parametrize("src_hw,res", [((480, 640), 240), ((360, 500), (240, 320)), ((480, 480), 480)])
def test_raw_frame_embeddings_are_bit_exact(src_hw, res):
    """uint8 HWC frames through the fused resize / normalise im2col give the embeddings of the preprocessed fp32 frames,
    bit for bit, square and non-square."""
    m, cfg, sd = _model("vit_small", 2, 2, "trained_like")
    rng = np.random.default_rng(src_hw[1])
    imgs = rng.integers(0, 256, (3, src_hw[0], src_hw[1], 3), dtype=np.uint8)
    hw = res if isinstance(res, tuple) else (res, res)
    u8 = torch.from_numpy(imgs).cuda()
    x = torch.from_numpy(np.stack([rect_ref.preprocess(im, hw) for im in imgs])).cuda()
    for kw in ({"n": 1}, {"n": 2}, {"n": 1, "avgpool": True}):
        e_u8 = m.embeddings(u8, resolution=res, **kw)
        e = m.embeddings(x, **kw)
        torch.cuda.synchronize()
        assert torch.equal(e_u8, e), kw


def test_wide_score_range():
    """q rows of the last block's qkv scaled so that the CLS query's scores reach +-128 log2 units, beyond the +-100 of
    attn_wide_901 in tools/gpu_check.py.  The CLS-only output stays finite and within the bars of the CPU reference
    on those weights, with the qkv GEMM's bf16 operands and outputs emulated (embeddings_ref.cls_block(bf16_qkv=True)),
    and no further from the all-fp32 reference than the full-size features path.  One block, so that the last block's
    input is the bf16x3 patch embedding: behind a bf16 block, the ~1e-2 relative error of the residual stream turns
    into score errors of several log2 units at this range, and the features path and this output both end near 7e-2
    of the fp32 reference (measured with two blocks)."""
    arch, nb, variant = "vit_small", 1, "trained_like"
    cfg = synthetic.make_config(arch, nb, 7)
    sd = synthetic.init_state_dict(cfg, 12, variant)
    x = synthetic.make_frames(2, 224, seed=12)
    d, hd, heads = cfg["embed_dim"], 64, cfg["num_heads"]
    p = f"dino.blocks.{nb - 1}."

    def max_score(sd):
        t = E.O.prepare_tokens(sd, x)
        y = torch.nn.functional.layer_norm(t, (d,), sd[p + "norm1.weight"], sd[p + "norm1.bias"], cfg["ln_eps"])
        w, b = sd[p + "attn.qkv.weight"], sd[p + "attn.qkv.bias"]
        q = torch.nn.functional.linear(y[:, :1], w[:d], b[:d]).reshape(2, 1, heads, hd).transpose(1, 2)
        k = torch.nn.functional.linear(y, w[d:2 * d], b[d:2 * d]).reshape(2, -1, heads, hd).transpose(1, 2)
        return float(((q @ k.transpose(-2, -1)) * hd ** -0.5 * np.log2(np.e)).abs().max())

    f = 128.0 / max_score(sd)
    sd = dict(sd)
    sd[p + "attn.qkv.weight"] = sd[p + "attn.qkv.weight"].clone()
    sd[p + "attn.qkv.bias"] = sd[p + "attn.qkv.bias"].clone()
    sd[p + "attn.qkv.weight"][:d] *= f
    sd[p + "attn.qkv.bias"][:d] *= f
    wide = max_score(sd)
    assert wide > 100, wide
    m, _, _ = _model(arch, nb, 12, variant, sd=sd)
    e = m.embeddings(x.cuda(), 1)
    full = m.features(x.cuda(), 1)[0, :, 0]
    torch.cuda.synchronize()
    ref32 = E.embeddings(sd, cfg, x, 1)
    err_cls, err_full = feature_errors(e.cpu(), ref32)[0], feature_errors(full.cpu(), ref32)[0]
    _record(case="emb_wide_range_fp32_ref", max_score_log2=wide, cls_only_max_rel=err_cls, features_max_rel=err_full)
    _check("emb_wide_range", e, E.cls_embedding_shortcut(sd, cfg, x, bf16_qkv=True), variant)
    assert err_cls <= 1.25 * err_full, (err_cls, err_full)


@pytest.mark.parametrize("arch,nb,cls_only", [("vit_small", 3, 21), ("vit_base", 4, 35)])
def test_launch_counts(arch, nb, cls_only):
    """The CLS-only call replaces the last block's attention pair (attention without row maxima + its redo) by one
    kernel and runs proj / MLP at M = B: one launch fewer than features(x, 1).  Every earlier requested block costs a
    row gather and the fp32 LayerNorm; the avgpool call is the feature pass with the pooling kernel in place of the
    LayerNorm."""
    m, cfg, sd = _model(arch, nb, 4, "reference_init")
    x = synthetic.make_frames(2, 64, seed=2).cuda()
    m.embeddings(x, 1)
    assert m.last_launch_count() == cls_only
    m.features(x, 1)
    n_feat = m.last_launch_count()
    assert cls_only < n_feat
    for n in range(1, nb + 2):
        m.embeddings(x, n)
        assert m.last_launch_count() == cls_only + 2 * (min(n, nb) - 1), n
    m.embeddings(x, 1, avgpool=True)
    assert m.last_launch_count() == n_feat


def test_embeddings_leave_the_other_paths_alone():
    """Forward label maps and features on the same handle are the same bits before and after embeddings calls, across
    a resolution switch."""
    m, cfg, sd = _model("vit_small", 3, 4, "trained_like")
    x = synthetic.make_frames(3, 240, seed=2).cuda()
    y = _frames(2, (480, 640), seed=5).cuda()
    lp0, low0, lab0 = m.infer(x, want_logprobs=True, want_lowres=True, want_labels=True)
    n_fwd = m.last_launch_count()
    f0 = m.features(x, 2)
    fy0 = m.features(y, 1)
    torch.cuda.synchronize()
    m.embeddings(y, 3)
    m.embeddings(x, 1, avgpool=True)
    m.embeddings(y, 1)
    lp1, low1, lab1 = m.infer(x, want_logprobs=True, want_lowres=True, want_labels=True)
    assert m.last_launch_count() == n_fwd
    m.embeddings(x, 2)
    f1 = m.features(x, 2)
    m.embeddings(x, 1)
    fy1 = m.features(y, 1)
    torch.cuda.synchronize()
    assert torch.equal(lp0, lp1) and torch.equal(low0, low1) and torch.equal(lab0, lab1)
    assert torch.equal(f0, f1) and torch.equal(fy0, fy1)


def test_errors():
    """n < 1, avgpool with more than one block, both C outputs NULL, a too small workspace, a bad resolution."""
    lib = _lib.load()
    m, cfg, sd = _model("vit_small", 2, 1, "reference_init")
    x = torch.zeros(1, 3, 64, 64, device="cuda")
    for bad in (0, -2):
        with pytest.raises(ValueError):
            m.embeddings(x, bad)
    with pytest.raises(ValueError, match="avgpool"):
        m.embeddings(x, 2, avgpool=True)
    with pytest.raises(ValueError, match="resolution"):
        m.embeddings(x, resolution=128)
    with pytest.raises(ValueError):
        m.embeddings(torch.zeros(1, 64, 64, 3, dtype=torch.uint8, device="cuda"), resolution=60)
    m.embeddings(x)                                             # handle, resolution 64 and workspace in place
    ws, hd = m._workspace, m._handle
    out = torch.full((2, 1, 384), 7.0, device="cuda")
    mean = torch.full((1, 384), 7.0, device="cuda")
    assert lib.dinoseg_embeddings(hd, x.data_ptr(), 1, 1, None, None, ws.data_ptr(), ws.numel(), None) != 0
    assert "NULL" in _lib.last_error(hd)
    assert lib.dinoseg_embeddings(hd, x.data_ptr(), 1, 0, out.data_ptr(), None, ws.data_ptr(), ws.numel(), None) != 0
    assert "n_last" in _lib.last_error(hd)
    assert lib.dinoseg_embeddings(hd, x.data_ptr(), 1, 1, out.data_ptr(), mean.data_ptr(), ws.data_ptr(), 1024,
                                  None) != 0
    assert "workspace too small" in _lib.last_error(hd)
    u8 = torch.zeros(1, 64, 64, 3, dtype=torch.uint8, device="cuda")
    mu, std = (C.c_float * 3)(0.5, 0.5, 0.5), (C.c_float * 3)(0.25, 0.25, 0.25)
    assert lib.dinoseg_embeddings_u8(hd, u8.data_ptr(), 1, 64, 64, mu, std, 1, None, None, ws.data_ptr(), ws.numel(),
                                     None) != 0
    assert lib.dinoseg_embeddings_u8(hd, u8.data_ptr(), 1, 0, 64, mu, std, 1, out.data_ptr(), None, ws.data_ptr(),
                                     ws.numel(), None) != 0
    torch.cuda.synchronize()
    assert (out == 7.0).all() and (mean == 7.0).all()           # nothing was enqueued
    h = C.c_void_p()
    cfg = _lib.DinosegCfg(384, 6, 1536, 1, 8, 28, 7, 200, 100, 0, 1e-6)
    assert lib.dinoseg_create(C.byref(cfg), 0, C.byref(h)) == 0
    try:
        assert lib.dinoseg_embeddings(h, x.data_ptr(), 1, 1, out.data_ptr(), None, ws.data_ptr(), ws.numel(), None) != 0
        assert "set_resolution" in _lib.last_error(h)
    finally:
        lib.dinoseg_destroy(h)
    # the C outputs alone: patch mean without CLS rows, CLS rows of two blocks with the patch mean
    assert lib.dinoseg_embeddings(hd, x.data_ptr(), 1, 1, None, mean.data_ptr(), ws.data_ptr(), ws.numel(), None) == 0
    assert lib.dinoseg_embeddings(hd, x.data_ptr(), 1, 2, out.data_ptr(), mean.data_ptr(), ws.data_ptr(), ws.numel(),
                                  None) == 0
    f = m.features(x, 2)
    torch.cuda.synchronize()
    assert torch.equal(out, f[:, :, 0])

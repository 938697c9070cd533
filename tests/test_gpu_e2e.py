"""End-to-end parity of the CUDA path (through the C-ABI, driven by the Python host in
dino_b200/model.py) on a real B200.

Against:  (1) tests/golden/*.npz — outputs of the UNMODIFIED reference on the same seeded weights and
frames (oracle/make_golden.py);  (2) the CPU oracle on fresh seeded inputs;  (3) size-independent
properties at BASELINE.json's full sizes (batch 64 @ 480 px): determinism, frame independence,
label map == replication of the low-res argmax, log-probs normalised.

Tolerances (bf16 tensor-core operands, fp32 accumulation / residual stream / LN / softmax / GELU):
  * per-patch log-probs: max-abs error <= TOL_ABS[variant], where 'reference_init' are the weights
    BASELINE.json names (near-uniform log-probs in [-2.4,-1.5]) and 'trained_like' is a stress
    variant with O(10)-magnitude logits, judged relative to the log-prob range;
  * label maps: >= 99.5 % of the pixels equal to the reference's for 'reference_init' weights (>= 98.5 % for
    the 'trained_like' stress weights), and EVERY differing patch must be a near-tie of the reference
    (top-2 log-prob margin below twice the max log-prob error);
  * argmax + replication on identical log-probs: bit-exact.
"""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN_CASES, ROOT, load_golden
from dino_b200 import DINOSeg, _lib, synthetic
from oracle import dinoseg_oracle as O

pytestmark = pytest.mark.gpu

TOL_ABS_REFINIT = 2e-3          # measured 3.5e-4 .. 7.5e-4 (SURVEY.md §7.3 expected 2e-3 for plain bf16 operands)
TOL_REL_TRAINED = 1.5e-2        # of the reference log-prob range (max - min)
MIN_LABEL_AGREEMENT = 0.995     # BASELINE.json north_star, for the random-init weights it names
MIN_LABEL_AGREEMENT_STRESS = 0.985   # 'trained_like' stress weights: many exact near-ties by construction


def _agreement_ok(got, ref):
    """>= 99.5 % of the patches equal; inputs with fewer than 400 patches may differ in at most 2
    (one near-tie there already costs more than 0.5 %)."""
    got, ref = np.asarray(got), np.asarray(ref)
    return float((got == ref).mean()) >= MIN_LABEL_AGREEMENT or int((got != ref).sum()) <= (2 if got.size < 400 else 0)
STATS_PATH = os.path.join(ROOT, "gpurun_out", "parity_stats.jsonl")


def _record(**kw):
    try:
        os.makedirs(os.path.dirname(STATS_PATH), exist_ok=True)
        with open(STATS_PATH, "a") as f:
            f.write(json.dumps(kw) + "\n")
    except OSError:
        pass


def _model(arch, n_blocks, seed, variant, n_classes=7, head="mlp"):
    cfg = synthetic.make_config(arch, n_blocks, n_classes, head=head)
    sd = synthetic.init_state_dict(cfg, seed, variant)
    m = DINOSeg(head=head, n_blocks=n_blocks, n_classes=n_classes, arch=arch)
    m.load_state_dict(sd, strict=True)
    return m.to("cuda:0"), cfg, sd


def _case(name):
    gd = load_golden(name)
    meta = gd["meta"]
    m, cfg, sd = _model(meta["arch"], meta["n_blocks"], meta["seed"], meta["variant"], meta["n_classes"],
                        meta.get("head", "mlp"))
    x = synthetic.make_frames(meta["batch"], meta["res"], meta["seed"])
    return gd, meta, m, cfg, sd, x


def _copy_buffer(m, name, shape, dtype):
    lib = _lib.load()
    out = torch.empty(shape, dtype=dtype, device="cuda:0")
    n = lib.dinoseg_copy_buffer(m._handle, name.encode(), out.data_ptr(), out.numel() * out.element_size(), None)
    assert n == out.numel() * out.element_size(), _lib.last_error(m._handle)
    torch.cuda.synchronize()
    return out.cpu()


def _compare_logprobs(tag, lp, ref, variant):
    err = np.abs(lp - ref)
    rng = float(ref.max() - ref.min())
    max_abs = float(err.max())
    rel = max_abs / rng
    mean_abs = float(err.mean())
    _record(case=tag, max_abs=max_abs, mean_abs=mean_abs, range=rng, rel_to_range=rel, variant=variant)
    if variant == "reference_init":
        # absolute bar for the near-uniform log-probs of the MLP head (range < 1); scaled with the range for heads
        # whose log-probs spread further (the 'linear' head: range ~4)
        assert max_abs <= TOL_ABS_REFINIT * max(1.0, rng), (tag, max_abs, rng)
    else:
        assert rel <= TOL_REL_TRAINED, (tag, max_abs, rng)
    return max_abs


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_against_reference_golden(name):
    """DINOSeg.forward + predict tail vs what the reference itself produced (pl_torch_modules.py:239-256,294-298)."""
    gd, meta, m, cfg, sd, x = _case(name)
    g = meta["res"] // 8
    lp, low, lab = m.infer(x.cuda(), want_logprobs=True, want_lowres=True, want_labels=True)
    torch.cuda.synchronize()
    lp, low, lab = lp.cpu().numpy(), low.cpu().numpy(), lab.cpu().numpy()
    assert lp.shape == gd["logprobs"].shape and np.isfinite(lp).all()
    max_abs = _compare_logprobs(name, lp, gd["logprobs"], meta["variant"])
    agree = float((low == gd["low"]).mean())
    _record(case=name, label_agreement=agree)
    assert agree >= (MIN_LABEL_AGREEMENT if meta["variant"] == "reference_init" else MIN_LABEL_AGREEMENT_STRESS), (name, agree)
    # every disagreeing patch must be a near-tie of the reference (top-2 margin below twice the error)
    srt = np.sort(gd["logprobs"], axis=1)
    margin = (srt[:, -1] - srt[:, -2]).reshape(low.shape)
    assert (margin[low != gd["low"]] <= 2 * max_abs + 1e-6).all()
    # output geometry and the replication itself (bit-exact on the kernel's own low-res map)
    p = 480 // g
    assert list(lab.shape) == gd["high_shape"].tolist() and lab.dtype == np.int64
    assert (lab == np.kron(low, np.ones((1, p, p), dtype=np.int64))).all()
    # the internal low-res argmax is the argmax of the returned log-probs (first max wins)
    assert (low.reshape(-1) == lp.argmax(1)).all()


@pytest.mark.parametrize("name", ["s8_nb1_240_refinit", "s8_nb3_240_b2_trained", "s8_nb2_224_trained", "b8_nb4_240_trained"])
def test_stage_rows_against_reference(name):
    """Positional table, prepare_tokens output and the residual stream after block 0 at sampled
    token rows (vision_transformer.py:202-235, :122-140)."""
    gd, meta, m, cfg, sd, x = _case(name)
    lib = _lib.load()
    B, g = meta["batch"], meta["res"] // 8
    N, D = g * g + 1, cfg["embed_dim"]
    rows = gd["rows"]
    xd = x.cuda()
    try:
        assert lib.dinoseg_set_debug_stop(m._ensure_handle() and m._handle, 1) == 0
        m.infer(xd)
        pos = _copy_buffer(m, "pos", (N, D), torch.float32).numpy()
        tok = _copy_buffer(m, "x", (B, N, D), torch.float32).numpy()
        assert lib.dinoseg_set_debug_stop(m._handle, 4) == 0
        m.infer(xd)
        blk0 = _copy_buffer(m, "x", (B, N, D), torch.float32).numpy()
    finally:
        lib.dinoseg_set_debug_stop(m._handle, 0)
    e_pos = float(np.abs(pos[rows] - gd["pos_rows"]).max())
    assert e_pos <= 2e-5 * max(1.0, float(np.abs(gd["pos_rows"]).max())), e_pos      # fp32 bicubic
    ref_tok, ref_blk = gd["tok_rows"], gd["blk0_rows"]
    e_tok = float(np.abs(tok[:, rows] - ref_tok).max()) / float(np.abs(ref_tok).max())
    e_blk = float(np.abs(blk0[:, rows] - ref_blk).max()) / float(np.abs(ref_blk).max())
    _record(case=name, pos_max_abs=e_pos, tokens_rel=e_tok, block0_rel=e_blk)
    assert e_tok <= 4e-3, e_tok       # one bf16-operand GEMM, K = 192
    assert e_blk <= 1e-2, e_blk       # + qkv, attention, proj, fc1, fc2


def test_argmax_replicate_bit_exact_on_reference_logprobs():
    """predict() tail on IDENTICAL log-probs: bit-exact (pl_torch_modules.py:295-298)."""
    lib = _lib.load()
    for name in ("s8_nb3_480_refinit", "s8_nb3_240_b2_trained", "s8_nb1_64_trained"):
        gd = load_golden(name)
        meta = gd["meta"]
        B, g = meta["batch"], meta["res"] // 8
        p = 480 // g
        lp = torch.from_numpy(gd["logprobs"]).cuda()
        low = torch.zeros(B, g, g, dtype=torch.uint8, device="cuda")
        lab = torch.zeros(B, g * p, g * p, dtype=torch.int64, device="cuda")
        assert lib.dinoseg_argmax_replicate(lp.data_ptr(), B, g, 7, p, low.data_ptr(), lab.data_ptr(), None) == 0
        torch.cuda.synchronize()
        assert (low.cpu().numpy() == gd["low"]).all()
        high = lab.cpu().numpy()
        assert list(high.shape) == gd["high_shape"].tolist()
        chk = [int(high.sum()), int((high * np.arange(high.size).reshape(high.shape) % 1000003).sum())]
        assert chk == gd["high_checksum"].tolist()


def test_predict_against_reference_golden():
    """DINOSeg.predict(PIL image) at 240 and 480 px vs the reference's predict on the same image."""
    from PIL import Image
    z = np.load(os.path.join(ROOT, "tests", "golden", "predict_s8_nb1.npz"))
    meta = json.loads(str(z["meta"]))
    m, cfg, sd = _model(meta["arch"], meta["n_blocks"], meta["seed"], meta["variant"])
    img = Image.fromarray(synthetic.make_image_u8(480, 640, meta["image_seed"]))
    for res in (240, 480):
        m.set_resolution(res)
        pred = m.predict(img)
        assert pred.shape == (480, 480) and pred.dtype == np.int64
        agree = float((pred == z[f"pred_{res}"]).mean())
        _record(case=f"predict_{res}", label_agreement=agree)
        assert agree >= MIN_LABEL_AGREEMENT, (res, agree)


@pytest.mark.parametrize("res,nb,batch", [(64, 1, 5), (224, 2, 1), (496, 1, 1), (8, 1, 3), (960, 1, 1)])
def test_against_oracle_edge_resolutions(res, nb, batch):
    """Ragged / extreme sizes: a single 128-key tile (64 px), the identity positional table
    (224 px, vision_transformer.py:205-206), an output that is not 480x480 (496 px -> 434x434,
    SURVEY.md §0), one patch per frame (8 px) and the 14401-token case (960 px)."""
    m, cfg, sd = _model("vit_small", nb, 11, "reference_init")
    x = synthetic.make_frames(batch, res, seed=res)
    g = res // 8
    p = 480 // g
    lp, low, lab = m.infer(x.cuda(), want_logprobs=True, want_lowres=True, want_labels=True)
    torch.cuda.synchronize()
    torch.set_num_threads(os.cpu_count() or 1)
    ref = O.forward(sd, cfg, x).numpy()
    ref_low, ref_high = O.labels_from_logprobs(torch.from_numpy(ref), batch, g)
    _compare_logprobs(f"oracle_{res}", lp.cpu().numpy(), ref, "reference_init")
    assert tuple(lab.shape) == tuple(ref_high.shape)
    assert _agreement_ok(low.cpu().numpy(), ref_low)
    # every disagreeing patch is a near-tie of the oracle (top-2 margin below twice the max error)
    srt = np.sort(ref, axis=1)
    margin = (srt[:, -1] - srt[:, -2]).reshape(ref_low.shape)
    err = float(np.abs(lp.cpu().numpy() - ref).max())
    assert (margin[low.cpu().numpy() != ref_low] <= 2 * err + 1e-6).all()
    assert (lab.cpu().numpy() == np.kron(low.cpu().numpy(), np.ones((1, p, p), dtype=np.int64))).all()


def test_full_size_batch_properties():
    """BASELINE.json configs[1] (batch 64, 480 px, 3 blocks): properties that need no reference."""
    m, cfg, sd = _model("vit_small", 3, 0, "reference_init")
    B, res, g = 64, 480, 60
    x = synthetic.make_frames(B, res, seed=1).cuda()
    lp, low, lab = m.infer(x, want_logprobs=True, want_lowres=True, want_labels=True)
    lp2, low2, _ = m.infer(x, want_logprobs=True, want_lowres=True)
    torch.cuda.synchronize()
    assert torch.equal(lp, lp2) and torch.equal(low, low2)                       # deterministic
    assert torch.isfinite(lp).all()
    assert (torch.logsumexp(lp.double(), dim=1).abs() <= 1e-5).all()             # log_softmax rows normalised
    assert torch.equal(low.reshape(-1).long(), lp.argmax(1))                     # argmax of its own log-probs
    up = low.long().repeat_interleave(8, dim=1).repeat_interleave(8, dim=2)
    assert torch.equal(lab, up)                                                  # np.kron(low, ones(8,8))
    # frames are independent: any sub-batch gives bit-identical results (no cross-frame leakage through
    # GEMM tiles that straddle frame boundaries, TMA zero-fill, or the attention key mask)
    for sl in (slice(0, 1), slice(5, 8), slice(61, 64)):
        lps, lows, _ = m.infer(x[sl].contiguous(), want_logprobs=True, want_lowres=True)
        torch.cuda.synchronize()
        n = g * g
        assert torch.equal(lps, lp[sl.start * n:sl.stop * n])
        assert torch.equal(lows, low[sl])
    # two frames of the batch against the CPU oracle
    torch.set_num_threads(os.cpu_count() or 1)
    idx = [0, 63]
    ref = O.forward(sd, cfg, x[idx].cpu()).numpy()
    got = torch.cat([lp[i * g * g:(i + 1) * g * g] for i in idx]).cpu().numpy()
    _compare_logprobs("full_size_b64_480", got, ref, "reference_init")
    ref_low, _ = O.labels_from_logprobs(torch.from_numpy(ref), 2, g)
    agree = float((low[idx].cpu().numpy() == ref_low).mean())
    _record(case="full_size_b64_480", label_agreement=agree)
    assert agree >= MIN_LABEL_AGREEMENT


@pytest.mark.parametrize("name,batch", [("s8_nb3_960_b2_refinit", 16), ("b8_nb4_480_b2_refinit", 32)])
def test_baseline_configs_4_and_5_at_full_batch(name, batch):
    """BASELINE.json configs[3] (ViT-S/8, 3 blocks, 960 px = 14401 tokens, batch 16) and configs[4]'s per-GPU shape
    (ViT-B/8, 4 blocks, 480 px, batch 32) at FULL batch: frames 0 and 1 of the batch are the two frames the unmodified
    reference was run on (tests/golden, oracle/make_golden.py; vision_transformer.py:80-107 at N = 14401, :307-311 +
    pl_torch_modules.py:108-124 for ViT-B), and any sub-batch must reproduce its slice of the full batch bit for bit
    (attention work-item plan, dual tail items and GEMM tiles change with the batch size; results must not)."""
    gd = load_golden(name)
    meta = gd["meta"]
    m, cfg, sd = _model(meta["arch"], meta["n_blocks"], meta["seed"], meta["variant"], meta["n_classes"])
    res, g = meta["res"], meta["res"] // 8
    n = g * g
    x = synthetic.make_frames(batch, res, meta["seed"])
    assert torch.equal(x[:2], synthetic.make_frames(2, res, meta["seed"]))       # the golden's frames
    xd = x.cuda()
    lp, low, lab = m.infer(xd, want_logprobs=True, want_lowres=True, want_labels=True)
    lp2, low2, _ = m.infer(xd, want_logprobs=True, want_lowres=True)
    torch.cuda.synchronize()
    assert torch.equal(lp, lp2) and torch.equal(low, low2) and torch.isfinite(lp).all()
    got = lp[:2 * n].cpu().numpy()
    max_abs = _compare_logprobs(name + f"_b{batch}", got, gd["logprobs"], meta["variant"])
    agree = float((low[:2].cpu().numpy() == gd["low"]).mean())
    _record(case=name + f"_b{batch}", label_agreement=agree)
    assert agree >= MIN_LABEL_AGREEMENT, (name, agree)
    srt = np.sort(gd["logprobs"], axis=1)
    margin = (srt[:, -1] - srt[:, -2]).reshape(gd["low"].shape)
    assert (margin[low[:2].cpu().numpy() != gd["low"]] <= 2 * max_abs + 1e-6).all()
    p = 480 // g
    assert torch.equal(lab, low.long().repeat_interleave(p, dim=1).repeat_interleave(p, dim=2))
    assert torch.equal(low.reshape(-1).long(), lp.argmax(1))
    for sl in (slice(0, 2), slice(batch // 2 - 1, batch // 2 + 2), slice(batch - 1, batch)):
        lps, lows, _ = m.infer(xd[sl].contiguous(), want_logprobs=True, want_lowres=True)
        torch.cuda.synchronize()
        assert torch.equal(lps, lp[sl.start * n:sl.stop * n]), sl
        assert torch.equal(lows, low[sl]), sl


def test_host_entry_point_matches_device_path():
    """dinoseg_predict_host (pinned host buffers in/out) == dinoseg_forward on device buffers, bit for bit."""
    m, cfg, sd = _model("vit_small", 2, 5, "trained_like")
    x = synthetic.make_frames(3, 240, seed=9)
    lab_dev = m.predict_batch(x.cuda(), output="labels")
    low_dev = m.predict_batch(x.cuda(), output="lowres")
    lab_host = m.predict_batch(x.pin_memory(), output="labels")
    low_host = m.predict_batch(x, output="lowres")            # pageable memory works too
    assert isinstance(lab_host, np.ndarray) and lab_host.dtype == np.int64
    assert (lab_host == lab_dev.cpu().numpy()).all() and (low_host == low_dev.cpu().numpy()).all()
    # the two ways of producing host label maps (GPU replication + D2H of the whole int64 maps, the default; low-res
    # D2H + expansion by the library's host threads) give the same bytes
    lib = _lib.load()
    assert lib.dinoseg_get_host_expand(m._handle) in (0, 1)   # automatic by default (host cores per rank)
    big = synthetic.make_frames(23, 240, seed=3)               # several chunks, ragged first / last chunk
    big_dev = m.predict_batch(big.cuda(), output="labels").cpu().numpy()
    for mode in (1, 0):
        assert lib.dinoseg_set_host_expand(m._handle, mode) == 0 and lib.dinoseg_get_host_expand(m._handle) == mode
        assert (m.predict_batch(x.pin_memory(), output="labels") == lab_host).all()
        assert (m.predict_batch(big.pin_memory(), output="labels") == big_dev).all()
    assert lib.dinoseg_set_host_expand(m._handle, -1) == 0


def test_folder_inference_matches_predict(tmp_path):
    """dt_segmentation/visualize.py-style folder inference (batched, pipelined) returns for every image exactly the map
    DINOSeg.predict(image) returns (reference visualize.py:36-54 calls predict once per image)."""
    from PIL import Image
    from dino_b200 import folder
    m, cfg, sd = _model("vit_small", 1, 7, "trained_like")
    m.set_resolution(240)
    sizes = [(480, 640)] * 5 + [(360, 500)] * 2 + [(480, 640)]
    for k, hw in enumerate(sizes):
        img = synthetic.make_image_u8(hw[0], hw[1], seed=50 + k)
        Image.fromarray(img).save(tmp_path / f"f{k:02d}.png")
    got = list(folder.predict_folder(m, str(tmp_path), batch_size=3))
    assert len(got) == len(sizes)
    assert [os.path.basename(p) for p, _, _ in got] == [os.path.basename(f) for f in folder.list_images(str(tmp_path))]
    for path, rgb, pred in got:
        want = m.predict(Image.open(path).convert("RGB"))
        assert pred.shape == (480, 480) and pred.dtype == np.int64 and (pred == want).all(), path
    # the drop-in script writes one overlay per image
    import dt_segmentation.visualize as V
    ck = tmp_path / "m.ckpt"
    torch.save({"state_dict": sd, "hyper_parameters": dict(head="mlp", n_blocks=1, n_classes=7)}, ck)
    assert V.inference(str(ck), str(tmp_path), str(tmp_path / "out"), resolution=240, batch_size=4) == len(sizes)
    assert sorted(os.listdir(tmp_path / "out")) == sorted(os.path.basename(p) for p, _, _ in got)
    with pytest.raises(RuntimeError, match="no CPU path"):
        V.inference(str(ck), str(tmp_path), str(tmp_path / "out2"), cpu=True)


@pytest.mark.parametrize("expand", [0, 1])
def test_async_host_submissions_match_the_synchronous_call(expand):
    """dinoseg_predict_host_submit / _wait: several batches in flight at once (they queue behind each other on the
    library's streams) give the bytes of one synchronous predict_batch call each, in both label-map modes (GPU
    replication + DMA, low-res D2H + host expansion); misuse is reported, not undefined."""
    lib = _lib.load()
    m, cfg, sd = _model("vit_small", 2, 5, "trained_like")
    m.set_resolution(240)
    xs = [synthetic.make_frames(n, 240, seed=20 + n).pin_memory() for n in (5, 23, 1, 12)]
    raw = torch.from_numpy(np.random.default_rng(3).integers(0, 256, (7, 480, 640, 3), dtype=np.uint8)).pin_memory()
    want = [m.predict_batch(x.cuda(), output="labels").cpu().numpy() for x in xs]
    want_raw = m.infer_u8(raw.cuda(), 240, want_logprobs=False, want_lowres=True)[1].cpu().numpy()
    assert lib.dinoseg_set_host_expand(m._handle, expand) == 0 and lib.dinoseg_get_host_expand(m._handle) == expand
    try:
        for _ in range(2):                                   # second round reuses tickets, lanes and staging buffers
            tickets = [m.predict_batch_async(x) for x in xs]                        # four submissions outstanding
            with pytest.raises(RuntimeError, match="outstanding"):
                m.predict_batch_async(xs[0])                                        # the fifth is refused
            got = [m.predict_wait(t) for t in reversed(tickets)][::-1]              # waiting out of order is fine
            for g_, w_ in zip(got, want):
                assert g_.dtype == np.int64 and (g_ == w_).all()
            t_raw = m.predict_batch_async(raw, resolution=240, output="lowres")
            t_f32 = m.predict_batch_async(xs[1])
            assert (m.predict_wait(t_f32) == want[1]).all()
            assert (m.predict_wait(t_raw) == want_raw).all()
            with pytest.raises(KeyError):
                m.predict_wait(t_raw)                                               # a ticket is good for one wait
        assert lib.dinoseg_predict_host_wait(m._handle, 12345) != 0 and "unknown ticket" in _lib.last_error(m._handle)
        assert lib.dinoseg_predict_host_wait(m._handle, 0) == 0                     # nothing outstanding: a no-op
    finally:
        lib.dinoseg_set_host_expand(m._handle, -1)


@pytest.mark.parametrize("hw,res", [((480, 640), 480), ((480, 640), 240), ((360, 500), 480), ((480, 480), 480)])
def test_gpu_preprocessing_is_bit_exact(hw, res):
    """uint8 frames -> (resize, normalise, im2col) on the GPU == the preprocessing oracle (= cv2.resize + fp32
    normalisation) followed by the fp32 path: identical log-probs, bit for bit (reference pl_torch_modules.py:33-41)."""
    from oracle import preproc_oracle as P
    m, cfg, sd = _model("vit_small", 1, 2, "trained_like")
    rng = np.random.default_rng(res + hw[1])
    imgs = rng.integers(0, 256, (3, hw[0], hw[1], 3), dtype=np.uint8)
    m.set_resolution(res)
    lp_u8, low_u8, _ = m.infer_u8(torch.from_numpy(imgs).cuda(), res, want_logprobs=True, want_lowres=True)
    x = torch.from_numpy(np.stack([P.preprocess(im, res) for im in imgs])).cuda()
    lp_f, low_f, _ = m.infer(x, want_logprobs=True, want_lowres=True)
    torch.cuda.synchronize()
    assert torch.equal(lp_u8, lp_f) and torch.equal(low_u8, low_f)
    # host entry point on raw frames == device path
    lab = m.predict_batch_u8(torch.from_numpy(imgs), res, output="lowres")
    assert (lab == low_f.cpu().numpy()).all()


@pytest.mark.parametrize("name", ["s8_nb1_240_refinit", "s8_nb3_240_b2_trained", "b8_nb4_240_refinit"])
def test_cls_attention_against_reference(name):
    """model.dino.get_last_selfattention(x)[b, :, 0, :] (the row visualize_attention.py:46-54 reads) vs the reference's
    (vision_transformer.py:273-280): rows are probability vectors; max error <= 1 % of the largest probability (measured
    0.15 - 0.5 %; 6 % for the peaked attention of the 'trained_like' stress weights, whose bf16 q/k rounding moves the
    logits by ~0.02: measured 5.2 %)."""
    gd, meta, m, cfg, sd, x = _case(name)
    att = m.dino.get_last_selfattention(x.cuda())
    torch.cuda.synchronize()
    n = (meta["res"] // 8) ** 2 + 1
    assert tuple(att.shape) == (meta["batch"], cfg["num_heads"], 1, n)
    got = att[:, :, 0, :].cpu().numpy()
    ref = gd["cls_attn"]
    assert np.abs(got.sum(-1) - 1.0).max() <= 1e-5
    err = float(np.abs(got - ref).max())
    _record(case=name, cls_attn_max_abs=err, cls_attn_ref_max=float(ref.max()))
    tol = 1e-2 if meta["variant"] == "reference_init" else 6e-2
    assert err <= tol * float(ref.max()), (err, float(ref.max()))


@pytest.mark.parametrize("res", [240, 24, 40])
def test_half_counts_match_oracle(res):
    """Controller-side reduction (SURVEY.md section 8(f)-4): left / right class pixel counts computed on the GPU from
    the low-res map equal a bincount over the halves of the int64 label map predict() returns (bit-exact; res 24 and
    40 have an odd patch grid, where the centre line cuts through a column of patches)."""
    m, cfg, sd = _model("vit_small", 1, 7, "trained_like")
    x = synthetic.make_frames(3, res, seed=9).cuda()
    _, low, lab = m.infer(x, want_logprobs=False, want_lowres=True, want_labels=True)
    got = m.half_counts(x).cpu().numpy()
    again = m.half_counts(low).cpu().numpy()
    ref = O.half_counts(lab.cpu().numpy(), cfg["n_classes"])
    assert got.dtype == np.int32 and got.shape == (3, 2, cfg["n_classes"])
    assert np.array_equal(got, ref) and np.array_equal(again, ref)
    assert int(got.sum()) == 3 * lab.shape[1] * lab.shape[2]


def test_fused_mlp_matches_unfused_path():
    """ViT-S runs fc1 -> GELU -> fc2 in one fused kernel; the unfused LN / fc1 / fc2 GEMM path (what ViT-B uses)
    must give the same log-probs up to bf16 rounding noise, and both must match the oracle."""
    lib = _lib.load()
    m, cfg, sd = _model("vit_small", 2, 3, "trained_like")
    x = synthetic.make_frames(2, 240, seed=4).cuda()
    a = m(x).clone()
    assert lib.dinoseg_set_fused_mlp(m._handle, 0) == 0
    b = m(x).clone()
    assert lib.dinoseg_set_fused_mlp(m._handle, 1) == 0
    c = m(x)
    torch.cuda.synchronize()
    assert torch.equal(a, c)
    ref = O.forward(sd, cfg, x.cpu())
    rng = float(ref.max() - ref.min())
    assert (a - b).abs().max().item() <= 5e-3 * rng
    assert (a.cpu() - ref).abs().max().item() <= TOL_REL_TRAINED * rng
    assert (b.cpu() - ref).abs().max().item() <= TOL_REL_TRAINED * rng


@pytest.mark.parametrize("variant,res,batch", [("reference_init", 240, 3), ("trained_like", 224, 2), ("trained_like", 64, 5),
                                               ("reference_init", 480, 9)])
def test_fused_head_matches_the_kernel_chain(variant, res, batch):
    """The one-kernel head (final LayerNorm -> layer_1 -> layer_2 -> layer_3 -> log_softmax -> argmax -> replication,
    csrc/head.cuh; reference vision_transformer.py:243, pl_torch_modules.py:117-124, :294-298) against the separate
    LayerNorm / GEMM / GEMM / tail kernels it replaces: both evaluate the head in bf16x3, so their log-probs agree far
    inside the bf16-vs-fp32 tolerance; label maps are the replication of each path's own argmax."""
    lib = _lib.load()
    m, cfg, sd = _model("vit_small", 2, 21, variant)
    x = synthetic.make_frames(batch, res, seed=res).cuda()
    g = res // 8
    p = 480 // g
    lp1, low1, lab1 = m.infer(x, want_logprobs=True, want_lowres=True, want_labels=True)
    n_fused = m.last_launch_count()
    assert lib.dinoseg_set_fused_head(m._handle, 0) == 0
    try:
        lp0, low0, lab0 = m.infer(x, want_logprobs=True, want_lowres=True, want_labels=True)
        n_chain = m.last_launch_count()
    finally:
        assert lib.dinoseg_set_fused_head(m._handle, 1) == 0
    torch.cuda.synchronize()
    assert n_chain == n_fused + 3                                  # LayerNorm + 2 GEMMs + tail -> 1 kernel
    rng = float(lp0.max() - lp0.min())
    d = float((lp1 - lp0).abs().max())
    _record(case=f"fused_head_{variant}_{res}", max_abs_vs_chain=d, range=rng)
    assert d <= 2e-4 * max(1.0, rng), (d, rng)
    assert torch.isfinite(lp1).all() and (torch.logsumexp(lp1.double(), dim=1).abs() <= 1e-5).all()
    assert torch.equal(low1.reshape(-1).long(), lp1.argmax(1))
    assert torch.equal(lab1, low1.long().repeat_interleave(p, dim=1).repeat_interleave(p, dim=2))
    differ = low1 != low0
    if differ.any():                                               # only where the chain's top-2 margin is below the difference
        srt = torch.sort(lp0, dim=1).values
        margin = (srt[:, -1] - srt[:, -2]).reshape(low0.shape)
        assert (margin[differ] <= 2 * d + 1e-7).all()
    # only one of the outputs requested
    _, low_only, _ = m.infer(x, want_logprobs=False, want_lowres=True)
    _, _, lab_only = m.infer(x, want_logprobs=False, want_labels=True)
    torch.cuda.synchronize()
    assert torch.equal(low_only, low1) and torch.equal(lab_only, lab1)


def test_bench_dumps_the_label_maps_of_its_timed_path(tmp_path):
    """bench.py --dump-outputs: the float32 copy of the int64 label maps of the last timed step, equal to what
    DINOSeg.infer returns for the bench's seeded weights (seed 0) and frames (seed 1); --steps is the number of timed steps."""
    import subprocess
    import sys
    dump = tmp_path / "dump"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--res", "240",
                        "--n-blocks", "1", "--batch", "3", "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(dump)],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    r = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    assert r["steps"] == 2 and r["gpu_launches"] % 2 == 0
    got = np.load(dump / "labels.npy")
    assert got.dtype == np.float32 and got.shape == (3, 480, 480)
    assert np.load(dump / "labels_frames.npy").tolist() == [0.0, 1.0, 2.0]
    m, cfg, sd = _model("vit_small", 1, 0, "reference_init")
    _, _, lab = m.infer(synthetic.make_frames(3, 240, seed=1).cuda(), want_logprobs=False, want_labels=True)
    assert np.array_equal(got, lab.cpu().numpy().astype(np.float32))


def test_weight_update_is_picked_up():
    """load_state_dict after the first forward re-packs the bf16 weights (no stale cache)."""
    m, cfg, sd = _model("vit_small", 1, 1, "reference_init")
    x = synthetic.make_frames(1, 64, seed=2).cuda()
    a = m(x).clone()
    sd2 = synthetic.init_state_dict(cfg, 2, "trained_like")
    m.load_state_dict(sd2)
    b = m(x)
    ref = O.forward(sd2, cfg, x.cpu())
    assert not torch.equal(a, b)
    assert (b.cpu() - ref).abs().max().item() <= TOL_REL_TRAINED * float(ref.max() - ref.min())


def test_error_paths():
    lib = _lib.load()
    m, cfg, sd = _model("vit_small", 1, 1, "reference_init")
    with pytest.raises(ValueError):
        m.infer(torch.zeros(1, 3, 60, 60, device="cuda"))          # resolution not a multiple of 8
    with pytest.raises(ValueError):
        m.infer(torch.zeros(1, 1, 64, 64, device="cuda"))          # grayscale: reference feeds 3 channels
    with pytest.raises(ValueError):
        m.infer(torch.zeros(1, 3, 64, 64))                          # frames on the CPU
    # raw C-ABI misuse returns an error code and a message, never crashes
    h = C.c_void_p()
    c = _lib.DinosegCfg(384, 6, 1536, 1, 8, 28, 7, 200, 100, 0, 1e-6)
    assert lib.dinoseg_create(C.byref(c), 0, C.byref(h)) == 0
    assert lib.dinoseg_set_resolution(h, 64, None) != 0 and "pos_embed" in _lib.last_error(h)
    x = torch.zeros(1, 3, 64, 64, device="cuda")
    ws = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
    assert lib.dinoseg_forward(h, x.data_ptr(), 1, None, None, None, ws.data_ptr(), ws.numel(), None) != 0
    bad = _lib.DinosegCfg(320, 5, 1280, 1, 8, 28, 7, 200, 100, 0, 1e-6)
    h2 = C.c_void_p()
    assert lib.dinoseg_create(C.byref(bad), 0, C.byref(h2)) != 0 and "embed_dim" in _lib.last_error(None)
    lib.dinoseg_destroy(h)
    # a correct handle with a too-small workspace
    m(x)
    assert lib.dinoseg_forward(m._handle, x.data_ptr(), 1, None, None, None, ws.data_ptr(), 1024, None) != 0
    assert "workspace too small" in _lib.last_error(m._handle)

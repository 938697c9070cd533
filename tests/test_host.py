"""Host-side checks that need no GPU: the C-ABI library loads and exports every symbol declared
in include/dinoseg.h, the Python surface mirrors the reference's (names, arguments, errors), the
product path never falls back to the CPU, and the frame sharding used for N > 1 GPUs is right
(world_size-2 gloo run)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from dino_b200 import DINOSeg, _lib, dist, synthetic
from dino_b200 import build as B


def _declared_symbols():
    with open(os.path.join(ROOT, "include", "dinoseg.h")) as f:
        src = f.read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(dinoseg_[a-z0-9_]+)\s*\(", src)))


def test_library_builds_and_exports_every_declared_symbol():
    path = B.build()
    assert os.path.exists(path)
    lib = ctypes.CDLL(path)
    names = _declared_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/dinoseg.h but not exported"
    assert sorted(_lib.SIGNATURES) == names, "ctypes prototypes and the header disagree"


def test_library_contains_blackwell_sass():
    """tcgen05 / TMA must be in the SASS of the shipped library (no mma.sync path)."""
    path = B.build()
    out = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True).stdout
    assert "UTCHMMA" in out or "UTCMMA" in out or "UTC" in out
    assert "UTMALDG" in out
    assert "LDTM" in out
    assert "HMMA" not in out.replace("UTCHMMA", "")
    assert "sm_100a" in subprocess.run(["cuobjdump", "-lelf", path], capture_output=True, text=True).stdout


def test_create_fails_without_gpu_instead_of_falling_back():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = _lib.load()
    cfg = _lib.DinosegCfg(384, 6, 1536, 1, 8, 28, 7, 200, 100, 0, 1e-6)
    h = ctypes.c_void_p()
    assert lib.dinoseg_create(ctypes.byref(cfg), 0, ctypes.byref(h)) != 0
    assert "no CUDA device" in _lib.last_error(None) or "CPU" in _lib.last_error(None)


def test_forward_on_cpu_model_raises():
    m = DINOSeg(head="mlp", n_blocks=1)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(1, 3, 64, 64))


def test_set_resolution_semantics():
    """pl_torch_modules.py:270-274."""
    m = DINOSeg(head="mlp", n_blocks=1)
    assert m.resolution == 480
    m.set_resolution(240)
    assert m.resolution == 240 and m.transforms.resolution == 240
    with pytest.raises(ValueError, match="Resolution should be a multiple of 8."):
        m.set_resolution(250)
    assert m.resolution == 240


def test_state_dict_keys_and_shapes_match_reference_inventory():
    """SURVEY.md §3.1 state-dict inventory (n_blocks=3, MLP head, 7 classes)."""
    m = DINOSeg(head="mlp", n_blocks=3, n_classes=7)
    sd = m.state_dict()
    ref = synthetic.init_state_dict(synthetic.make_config("vit_small", 3, 7))
    assert list(sd.keys()) == list(ref.keys()) or sorted(sd.keys()) == sorted(ref.keys())
    for k, v in ref.items():
        assert tuple(sd[k].shape) == tuple(v.shape), k
    assert sd["dino.pos_embed"].shape == (1, 785, 384)
    assert sum(v.numel() for v in sd.values()) == 5_796_091 or abs(sum(v.numel() for v in sd.values()) - 5.80e6) < 2e4


def test_load_from_checkpoint_roundtrip(tmp_path):
    """PL-style checkpoint: {'state_dict', 'hyper_parameters'} (SURVEY.md §5); hyper-parameters
    of the training side (optimizer class, loggers) are accepted and ignored."""
    cfg = synthetic.make_config("vit_small", 2, 5)
    sd = synthetic.init_state_dict(cfg, 3, "trained_like")
    hp = dict(data_path="d", write_path="w", class_names=None, head="mlp", n_blocks=2, batch_size=1, lr=1e-6,
              optimizer=torch.optim.AdamW, freeze_backbone=True, max_epochs=200, patience=10, grayscale=False,
              n_classes=5, pretrain_on_sim=False, comet_logger=None, augmented=True, random_init=False, backbone="vit")
    path = tmp_path / "m.ckpt"
    torch.save({"state_dict": sd, "hyper_parameters": hp, "epoch": 3}, path)
    m = DINOSeg.load_from_checkpoint(str(path))
    assert m.n_blocks == 2 and m.n_classes == 5 and m.head == "mlp"
    for k, v in m.state_dict().items():
        assert torch.equal(v, sd[k]), k
    bad = dict(sd)
    bad.pop("clf.layer_3.bias")
    torch.save({"state_dict": bad, "hyper_parameters": hp}, path)
    with pytest.raises(RuntimeError):
        DINOSeg.load_from_checkpoint(str(path))


def test_load_from_checkpoint_with_classes_of_packages_that_are_not_installed(tmp_path):
    """A real PL checkpoint pickles objects of the training environment (e.g. a comet logger): the tolerant unpickler
    (model.py::_TolerantUnpickler) replaces classes that cannot be resolved by inert placeholders and the weights still
    load; a file that is simply corrupt raises the ORIGINAL error instead of being masked by the retry."""
    import importlib
    import types
    cfg = synthetic.make_config("vit_small", 1, 7)
    sd = synthetic.init_state_dict(cfg, 4, "reference_init")
    mod = types.ModuleType("some_training_only_package")
    class CometLogger:                                   # lives in a module that will not exist at load time
        def __init__(self):
            self.key = "secret"
    CometLogger.__module__ = "some_training_only_package"
    CometLogger.__qualname__ = "CometLogger"
    mod.CometLogger = CometLogger
    sys.modules["some_training_only_package"] = mod
    path = tmp_path / "pl.ckpt"
    try:
        hp = dict(head="mlp", n_blocks=1, n_classes=7, comet_logger=CometLogger(), data_path="d", write_path="w")
        torch.save({"state_dict": sd, "hyper_parameters": hp, "callbacks": {"logger": CometLogger()}}, path)
    finally:
        del sys.modules["some_training_only_package"]
    with pytest.raises(ModuleNotFoundError):             # the plain load cannot resolve the class ...
        torch.load(path, map_location="cpu", weights_only=False)
    m = DINOSeg.load_from_checkpoint(str(path))          # ... the drop-in loader can
    assert m.n_blocks == 1 and m.head == "mlp"
    for k, v in m.state_dict().items():
        assert torch.equal(v, sd[k]), k
    assert type(m.comet_logger).__name__ == "CometLogger" and not hasattr(m.comet_logger, "key")   # inert placeholder
    # a corrupt file is reported as such (no tolerant retry, no placeholder objects)
    bad = tmp_path / "corrupt.ckpt"
    bad.write_bytes(path.read_bytes()[:2000])
    with pytest.raises(Exception) as ei:
        DINOSeg.load_from_checkpoint(str(bad))
    assert not isinstance(ei.value, (KeyError, TypeError)), ei.value


def test_unsupported_variants_fail_loudly():
    with pytest.raises(NotImplementedError):
        DINOSeg(head="mlp", backbone="cnn1")
    with pytest.raises(ValueError):
        DINOSeg(head="conv")
    lin = DINOSeg(head="linear", n_classes=5)          # reference default head (pl_torch_modules.py:145, :127-138)
    assert sorted(k for k in lin.state_dict() if k.startswith("clf.")) == ["clf.layer_1.bias", "clf.layer_1.weight"]
    assert lin.state_dict()["clf.layer_1.weight"].shape == (5, 384)
    with pytest.raises(NotImplementedError):
        DINOSeg(head="mlp").fit()


def test_drop_in_import_path():
    import dt_segmentation
    assert dt_segmentation.DINOSeg is DINOSeg
    assert callable(dt_segmentation.parse_class_names)


def test_transforms_restatement():
    """Resize(INTER_LINEAR) -> Normalize(ImageNet) -> CHW (pl_torch_modules.py:33-41)."""
    from dino_b200.transforms import get_transforms, IMAGENET_MEAN, IMAGENET_STD
    img = synthetic.make_image_u8(480, 640, 3)
    out = get_transforms(240)(image=img)["image"]
    assert out.shape == (3, 240, 240) and out.dtype == torch.float32
    same = get_transforms(480)(image=img[:, :480])["image"]
    ref = (img[:, :480].astype(np.float32) / 255.0 - np.array(IMAGENET_MEAN, np.float32)) / np.array(IMAGENET_STD, np.float32)
    assert np.abs(same.numpy() - ref.transpose(2, 0, 1)).max() < 1e-5


@pytest.mark.parametrize("total,world", [(512, 8), (64, 1), (10, 4), (3, 8), (0, 2)])
def test_shard_range_partitions(total, world):
    spans = [dist.shard_range(total, r, world) for r in range(world)]
    assert spans[0][0] == 0 and spans[-1][1] == total
    for (a0, a1), (b0, b1) in zip(spans, spans[1:]):
        assert a1 == b0 and a1 >= a0
    sizes = [b - a for a, b in spans]
    assert max(sizes) - min(sizes) <= 1


_GLOO_WORKER = r"""
import os, sys, json
sys.path.insert(0, sys.argv[1])
import torch
from dino_b200 import dist as D, synthetic
rank, local, world = D.init(backend="gloo")
lo, hi = D.shard_range(10, rank, world)
frames = synthetic.make_frames(10, 16, seed=1)[lo:hi]
D.barrier()
s = D.sum_over_ranks(float(frames.double().sum()))
n = D.sum_over_ranks(hi - lo)
m = D.max_over_ranks(float(rank + 1))
if rank == 0:
    tot = float(synthetic.make_frames(10, 16, seed=1).double().sum())
    print(json.dumps({"ok": abs(s - tot) < 1e-6 and n == 10 and m == world, "world": world}))
D.barrier(); D.shutdown()
"""


def test_two_rank_gloo_sharding(tmp_path):
    """N > 1 path on CPU: world_size 2, gloo, frames sharded by rank, no data-path collective."""
    script = tmp_path / "w.py"
    script.write_text(_GLOO_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29731", OMP_NUM_THREADS="1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29731", str(script), ROOT]
    p = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=240)
    assert p.returncode == 0, p.stderr[-2000:]
    line = [l for l in p.stdout.splitlines() if l.startswith("{")][-1]
    import json
    r = json.loads(line)
    assert r["ok"] and r["world"] == 2


def test_bench_reference_arm_contract(tmp_path):
    """`bench.py --impl reference` prints one JSON line with the reference-arm keys (tiny config); --dump-outputs writes
    the label map of its last timed step (frame 0 of the batch)."""
    import json
    from oracle import dinoseg_oracle as O
    dump = tmp_path / "dump"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "1", "--res", "64", "--n-blocks", "1", "--batch", "2", "--dump-outputs", str(dump)],
                       capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr[-2000:]
    r = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    assert r["impl"] == "reference" and r["unit"] == "frames/s" and r["value"] > 0
    assert r["cpu_baseline"]["kind"] == "port" and r["cpu_baseline"]["cores"] >= 1
    assert r["e2e"]["h2d_bytes_per_step"] == 0 and r["e2e"]["value"] == r["value"]
    got = np.load(dump / "labels.npy")
    assert got.dtype == np.float32 and got.shape == (1, 480, 480)
    assert np.load(dump / "labels_frames.npy").tolist() == [0.0]
    cfg = synthetic.make_config("vit_small", 1, 7)
    lp = O.forward(synthetic.init_state_dict(cfg, 0, "reference_init"), cfg, synthetic.make_frames(1, 64, seed=1),
                   frame_chunk=1)
    assert np.array_equal(got, O.labels_from_logprobs(lp, 1, 8)[1].astype(np.float32))


def test_bench_dump_samples_a_fixed_set_of_frames_over_budget(tmp_path):
    """--dump-outputs keeps under its byte budget: a batch that does not fit is cut to a seeded sample of frames (the same
    in every run, listed in <name>_frames.npy); a batch that fits is written whole."""
    import importlib
    sys.path.insert(0, ROOT)
    bench = importlib.import_module("bench")
    labels = torch.arange(10 * 4 * 4, dtype=torch.int64).reshape(10, 4, 4)
    budget = 4096 + 8 * 10 + 3 * 4 * 4 * 4                       # headers and index + three float32 frames
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), "labels", labels, budget)
    keep = np.load(tmp_path / "a" / "labels_frames.npy")
    got = np.load(tmp_path / "a" / "labels.npy")
    assert keep.dtype == np.float64 and len(keep) == 3 and (np.diff(keep) > 0).all()
    assert got.dtype == np.float32 and np.array_equal(got, labels.numpy()[keep.astype(int)].astype(np.float32))
    assert np.array_equal(np.load(tmp_path / "b" / "labels_frames.npy"), keep)
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= budget
    bench.dump_outputs(str(tmp_path / "c"), "labels", labels, 1 << 20)
    assert np.array_equal(np.load(tmp_path / "c" / "labels.npy"), labels.numpy().astype(np.float32))
    assert np.load(tmp_path / "c" / "labels_frames.npy").tolist() == list(range(10))


@pytest.mark.parametrize("g,p,offset", [(60, 8, 0), (30, 16, 0), (62, 7, 0), (3, 160, 0), (1, 480, 0), (5, 96, 8)])
def test_host_label_expansion_matches_np_kron(g, p, offset):
    """The host-side label expansion of the library (used by dinoseg_set_host_expand) == np.kron(low, ones((p, p))),
    reference pl_torch_modules.py:297-298 - including a 7-pixel replication (odd row length: no streaming stores) and
    an output buffer that is only 8-byte aligned."""
    import ctypes as C
    from dino_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(g * 1000 + p)
    low = rng.integers(0, 256, size=(3, g, g), dtype=np.uint8)
    w = g * p
    buf = np.full(3 * w * w + 2, -7, dtype=np.int64)
    out = buf[offset // 8: offset // 8 + 3 * w * w].reshape(3, w, w)
    rc = lib.dinoseg_expand_labels_host(low.ctypes.data_as(C.c_void_p), 3, g, p, out.ctypes.data_as(C.c_void_p))
    assert rc == 0
    ref = np.stack([np.kron(low[b].astype(np.int64), np.ones((p, p), dtype=np.int64)) for b in range(3)])
    assert np.array_equal(out, ref)
    assert (buf[3 * w * w + offset // 8:] == -7).all()


@pytest.mark.parametrize("B,H,N", [(64, 6, 3601), (1, 6, 3601), (3, 6, 785), (2, 6, 901), (1, 1, 65), (3, 1, 129),
                                   (5, 3, 300), (1, 12, 3601), (7, 1, 1), (2, 12, 14401)])
def test_attention_work_items_cover_every_query_tile_once(B, H, N):
    """The attention kernel's work-item plan (regular items = two query tiles of one head, dual tail items = the lone
    last tiles of two heads, single tail item for an odd number of heads): every (frame*H + head, query tile) is
    covered exactly once, and a dual item directly follows the regular items of its two heads."""
    import ctypes as C
    from dino_b200 import _lib
    lib = _lib.load()
    n = lib.dinoseg_debug_attn_items(B, H, N, None, 0)
    q_tiles = (N + 127) // 128
    bh = B * H
    assert n == bh * (q_tiles // 2) + ((bh + 1) // 2 if q_tiles % 2 else 0)
    buf = np.zeros((n, 6), dtype=np.int32)
    assert lib.dinoseg_debug_attn_items(B, H, N, buf.ctypes.data_as(C.c_void_p), n) == n
    seen = {}
    for i, (bh0, q0, bh1, q1, act1, dual) in enumerate(buf.tolist()):
        assert 0 <= bh0 < bh and q0 % 128 == 0 and 0 <= q0 < N
        seen[(bh0, q0 // 128)] = seen.get((bh0, q0 // 128), 0) + 1
        if act1:
            assert 0 <= bh1 < bh and q1 % 128 == 0 and 0 <= q1 < N
            seen[(bh1, q1 // 128)] = seen.get((bh1, q1 // 128), 0) + 1
        assert bool(dual) == (bool(act1) and bh0 != bh1)
        if dual:                                     # K/V locality: the item before it belongs to one of its heads
            assert q0 == q1 == (q_tiles // 2) * 256 and bh1 == bh0 + 1
            if q_tiles > 1:
                assert buf[i - 1][0] == bh1
    assert len(seen) == bh * q_tiles and all(v == 1 for v in seen.values())


def test_bench_stall_watchdog_ends_the_run():
    """A run that does not finish inside --stall-limit prints an error line and exits with code 3 instead of hanging."""
    import json
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "50",
                        "--warmup", "1", "--stall-limit", "2"], capture_output=True, text=True, timeout=120)
    assert p.returncode == 3, (p.returncode, p.stderr[-500:])
    r = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    assert "stalled" in r["error"]


def test_bench_never_retries_a_stalled_run():
    """The B200 arm has no supervisor: a run that stalls ends ONCE with the error line and exit code 3 (a retry in the
    measurement harness would hide exactly the failure a user would hit), and the process that measures is the
    process that was started (no child, no second attempt)."""
    import json
    env = dict(os.environ, DINOSEG_BENCH_TEST_STALL="1")
    env.pop("WORLD_SIZE", None)
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--stall-limit", "1.5"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert p.returncode == 3, (p.returncode, p.stderr[-500:])
    assert p.stderr.count("no result after") == 1 and "retry" not in p.stderr
    r = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    assert "stalled" in r["error"] and "attempt" not in r
    with open(os.path.join(ROOT, "bench.py")) as f:
        src = f.read()
    assert "def supervise" not in src and "CDLL" not in src


def test_bench_default_batch_follows_baseline_configs():
    """configs[1]: 64 frames on one GPU; configs[2]: 512 frames sharded across 2 / 4 / 8 GPUs (strong scaling)."""
    import importlib
    sys.path.insert(0, ROOT)
    bench = importlib.import_module("bench")
    old_argv, old_ws = sys.argv, os.environ.get("WORLD_SIZE")
    try:
        for world, flags, want in ((1, [], (64, "weak")), (2, [], (256, "strong")), (4, [], (128, "strong")),
                                   (8, [], (64, "strong")), (8, ["--batch", "64"], (64, "weak")),
                                   (4, ["--global-batch", "512"], (128, "strong")), (1, ["--global-batch", "512"], (512, "strong"))):
            os.environ["WORLD_SIZE"] = str(world)
            sys.argv = ["bench.py"] + flags
            a = bench.parse_args()
            assert (a.batch, a.scaling) == want, (world, flags, a.batch, a.scaling)
    finally:
        sys.argv = old_argv
        if old_ws is None:
            os.environ.pop("WORLD_SIZE", None)
        else:
            os.environ["WORLD_SIZE"] = old_ws


def test_bench_reads_the_attention_traffic_from_profiles():
    """roofline.traffic comes from the committed ncu summary, not from a literal in bench.py."""
    import importlib
    sys.path.insert(0, ROOT)
    bench = importlib.import_module("bench")
    traffic, src, _ = bench.ncu_attention_traffic()
    assert src is not None and src.startswith("profiles/") and 5e8 < traffic < 1e9, (traffic, src)


def test_folder_inference_host_logic(tmp_path):
    """dino_b200.folder: the reference's traversal order (visualize.py:36-37: *.jpg then *.png), batches of consecutive
    equal-size frames, results in input order with two batches in flight, and the overlay renderer."""
    from PIL import Image
    from dino_b200 import folder
    rng = np.random.default_rng(0)
    names = ["b.png", "a.jpg", "c.jpg", "d.png", "notes.txt"]
    for n in names[:-1]:
        Image.fromarray(rng.integers(0, 256, (48, 64, 3), dtype=np.uint8)).save(tmp_path / n)
    (tmp_path / names[-1]).write_text("x")
    files = folder.list_images(str(tmp_path))
    assert [os.path.splitext(f)[1] for f in files] == [".jpg", ".jpg", ".png", ".png"]
    assert folder.plan_batches([(4, 4)] * 5 + [(2, 2)] + [(4, 4)] * 2, 3) == [[0, 1, 2], [3, 4], [5], [6, 7]]

    class FakeModel:                                  # records the batches, answers with the frame's mean colour class
        resolution = 480

        def __init__(self):
            self.batches, self.results, self.max_in_flight = [], {}, 0

        def predict_batch_async(self, frames, resolution=None, output="labels"):
            assert frames.dtype == torch.uint8 and frames.dim() == 4 and frames.shape[3] == 3
            t = len(self.batches) + 1
            self.batches.append(tuple(frames.shape))
            self.results[t] = np.stack([np.full((4, 4), int(f.float().mean()) % 7, dtype=np.int64) for f in frames])
            self.max_in_flight = max(self.max_in_flight, len(self.results))
            return t

        def predict_wait(self, t):
            return self.results.pop(t)

    imgs = [np.full((8, 8, 3), v, dtype=np.uint8) for v in (10, 20, 30, 40, 50)] + [np.full((6, 8, 3), 60, dtype=np.uint8)] + \
           [np.full((8, 8, 3), 70, dtype=np.uint8)]
    fm = FakeModel()
    out = list(folder.predict_images(fm, iter(imgs), batch_size=2))
    assert [int(o[0, 0]) for o in out] == [v % 7 for v in (10, 20, 30, 40, 50, 60, 70)]     # input order
    assert fm.batches == [(2, 8, 8, 3), (2, 8, 8, 3), (1, 8, 8, 3), (1, 6, 8, 3), (1, 8, 8, 3)]
    assert fm.max_in_flight == 2
    with pytest.raises(ValueError):
        list(folder.predict_images(fm, [np.zeros((8, 8), dtype=np.uint8)]))
    pred = np.zeros((480, 480), dtype=np.int64)
    pred[:100] = 3
    ov = folder.overlay(pred, imgs[0].repeat(10, axis=0).repeat(10, axis=1))
    assert ov.shape == (480, 480, 3) and ov.dtype == np.uint8
    assert (ov[200:] == 10).all() and not (ov[:100] == 10).all()                               # class 0 keeps the grey image
    assert folder.label_colormap()[:4].tolist() == [[0, 0, 0], [128, 0, 0], [0, 128, 0], [128, 128, 0]]


def test_host_worker_pool_survives_a_failing_thread_creation():
    """std::thread creation can fail (EAGAIN: pids / nproc limit).  A partial failure keeps the smaller pool - it must not
    unwind with joinable threads (std::terminate) - and a failure of the very first thread is reported to the caller, who
    falls back to the DMA path (dinoseg_api.cu: HostPool, predict_host_submit_impl)."""
    lib = _lib.load()
    assert lib.dinoseg_debug_host_pool(6, -1) == 6          # all threads, all tasks ran
    assert lib.dinoseg_debug_host_pool(6, 3) == 3           # threads 0..2 exist and do all the work
    assert lib.dinoseg_debug_host_pool(6, 1) == 1
    assert lib.dinoseg_debug_host_pool(6, 0) == 0           # no thread at all: the caller's fallback


def test_product_code_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under dino_b200/ or dt_segmentation/ may use it."""
    for pkg in ("dino_b200", "dt_segmentation"):
        for dp, _, files in os.walk(os.path.join(ROOT, pkg)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h")):
                    with open(os.path.join(dp, f)) as fh:
                        src = fh.read()
                    assert not re.search(r"^\s*(import|from)\s+oracle\b", src, flags=re.M), f
                    assert "dinoseg_oracle" not in src, f

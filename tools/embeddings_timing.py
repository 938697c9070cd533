#!/usr/bin/env python
"""Image embeddings against the n = 1 feature pass at the bench shapes (ViT-S/8 3 blocks 480 px batch 64, ViT-B/8
4 blocks 480 px batch 32): milliseconds per call of dinoseg_features (n_last = 1) and dinoseg_embeddings (CLS rows of
the last 1 or n_blocks blocks, or the CLS row with the patch mean), the arms alternating call by call in one process
(CUDA events around each call, 3 warm-up rounds, 20 timed rounds, median), then one profiled call per arm for the
per-kind kernel times (profile_enable).  Prints one JSON line with the device name and power limit, and writes it to
--out if given."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from dino_b200 import DINOSeg, _lib, synthetic  # noqa: E402

SHAPES = [("vit_small", 3, 480, 64), ("vit_base", 4, 480, 32)]
WARMUP, STEPS = 3, 20


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except Exception:
        return None


def run_shape(arch, nb, res, batch):
    lib = _lib.load()
    cfg = synthetic.make_config(arch, nb, 7)
    m = DINOSeg(head="mlp", n_blocks=nb, n_classes=7, arch=arch)
    m.load_state_dict(synthetic.init_state_dict(cfg, 0, "reference_init"), strict=True)
    m = m.to("cuda:0")
    x = synthetic.make_frames(batch, res, seed=1).cuda()
    m.features(x, 1)                                       # handle, weights, resolution, workspace
    h, ws, stream = m._handle, m._workspace, m._stream()
    g, d = res // 8, cfg["embed_dim"]
    feats = torch.empty((1, batch, g * g + 1, d), dtype=torch.float32, device="cuda")
    cls = torch.empty((nb, batch, d), dtype=torch.float32, device="cuda")
    mean = torch.empty((batch, d), dtype=torch.float32, device="cuda")

    def features():
        return lib.dinoseg_features(h, x.data_ptr(), batch, 1, feats.data_ptr(), ws.data_ptr(), ws.numel(), stream)

    def embeddings(n, avgpool=False):
        return lambda: lib.dinoseg_embeddings(h, x.data_ptr(), batch, n, cls.data_ptr(),
                                              mean.data_ptr() if avgpool else None, ws.data_ptr(), ws.numel(), stream)

    arms = {"features_n1": features, "embeddings_n1": embeddings(1)}
    if arch == "vit_small":
        arms[f"embeddings_n{nb}"] = embeddings(nb)
    arms["embeddings_n1_avgpool"] = embeddings(1, True)
    launches = {}
    for name, fn in arms.items():
        assert fn() == 0, _lib.last_error(h)
        launches[name] = m.last_launch_count()
    times = {name: [] for name in arms}
    for step in range(WARMUP + STEPS):
        for name, fn in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            assert fn() == 0, _lib.last_error(h)
            e1.record()
            e1.synchronize()
            if step >= WARMUP:
                times[name].append(e0.elapsed_time(e1))
    kinds = {}
    for name, fn in arms.items():
        m.profile_enable(True)
        assert fn() == 0, _lib.last_error(h)
        torch.cuda.synchronize()
        kinds[name] = {k: [round(ms, 4), cnt] for k, (ms, cnt) in m.profile_read().items()}
        m.profile_enable(False)
    out = {}
    for name in arms:
        med = statistics.median(times[name])
        out[name] = {"ms_median": round(med, 4), "ms_min": round(min(times[name]), 4),
                     "ms_max": round(max(times[name]), 4), "frames_per_s": round(batch / (med / 1e3), 1),
                     "launches": launches[name], "kernel_ms_by_kind": kinds[name]}
    base = out["features_n1"]["ms_median"]
    return {"arch": arch, "n_blocks": nb, "res": res, "batch": batch, "arms": out,
            "time_vs_features_n1": {k: round(v["ms_median"] / base, 4) for k, v in out.items()}}


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("embeddings_timing.py needs a GPU")
    line = json.dumps({"device": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(), "warmup": WARMUP,
                       "steps": STEPS, "shapes": [run_shape(*s) for s in SHAPES]})
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

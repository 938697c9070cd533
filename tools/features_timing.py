#!/usr/bin/env python
"""Backbone-feature pass against the segmentation forward at the bench shapes (ViT-S/8 3 blocks 480 px batch 64,
ViT-B/8 4 blocks 480 px batch 32): frames/s of dinoseg_forward (int64 label maps, as bench.py times it) and of
dinoseg_features with n_last = 1 and n_last = n_blocks, the three arms alternating step by step in one process
(CUDA events around each call, 3 warm-up rounds, 20 timed rounds), then one profiled call per arm for the per-kind
kernel times (profile_enable).  Prints one JSON line with the device name and power limit."""
import ctypes as C
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
    m.set_resolution(res)
    x = synthetic.make_frames(batch, res, seed=1).cuda()
    m.infer(x, want_logprobs=False, want_labels=True)     # handle, weights, resolution, workspace
    h, ws, stream = m._handle, m._workspace, m._stream()
    g, d = res // 8, cfg["embed_dim"]
    labels = torch.empty((batch, g * (480 // g), g * (480 // g)), dtype=torch.int64, device="cuda")
    feats = torch.empty((nb, batch, g * g + 1, d), dtype=torch.float32, device="cuda")

    def forward():
        return lib.dinoseg_forward(h, x.data_ptr(), batch, None, None, labels.data_ptr(), ws.data_ptr(), ws.numel(), stream)

    def features(n):
        return lambda: lib.dinoseg_features(h, x.data_ptr(), batch, n, feats.data_ptr(), ws.data_ptr(), ws.numel(), stream)

    arms = {"forward": forward, "features_n1": features(1), f"features_n{nb}": features(nb)}
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
    res_arms = {}
    for name in arms:
        med = statistics.median(times[name])
        res_arms[name] = {"frames_per_s": round(batch / (med / 1e3), 1), "ms_median": round(med, 4),
                          "ms_min": round(min(times[name]), 4), "ms_max": round(max(times[name]), 4),
                          "launches": launches[name], "kernel_ms_by_kind": kinds[name]}
    # n_last = n_blocks runs n_blocks - 1 more fp32 LayerNorms than n_last = 1 and otherwise the same kernels
    ln1, ln_all = kinds["features_n1"]["layernorm"], kinds[f"features_n{nb}"]["layernorm"]
    fp32_ln_ms = round((ln_all[0] - ln1[0]) / (ln_all[1] - ln1[1]), 4) if ln_all[1] > ln1[1] else None
    fp32_ln_bytes = batch * (g * g + 1) * d * 8 + 2 * d * 4      # fp32 stream in, fp32 features out
    return {"arch": arch, "n_blocks": nb, "res": res, "batch": batch, "arms": res_arms,
            "features_n1_vs_forward": round(res_arms["features_n1"]["frames_per_s"] / res_arms["forward"]["frames_per_s"], 4),
            "fp32_layernorm_ms": fp32_ln_ms, "fp32_layernorm_bytes": fp32_ln_bytes,
            "fp32_layernorm_tb_per_s": round(fp32_ln_bytes / (fp32_ln_ms * 1e-3) / 1e12, 2) if fp32_ln_ms else None}


def main():
    if not torch.cuda.is_available():
        raise SystemExit("features_timing.py needs a GPU")
    out = {"device": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(), "warmup": WARMUP, "steps": STEPS,
           "shapes": [run_shape(*s) for s in SHAPES]}
    print(json.dumps(out))


if __name__ == "__main__":
    main()

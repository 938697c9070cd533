#!/usr/bin/env python
"""Non-square frames against square ones at the bench model (ViT-S/8, 3 blocks): frames/s and tokens/s of
dinoseg_forward (low-res maps: label maps exist for square frames only) and of dinoseg_features with n_last = 1, at
480x640 (4801 tokens) next to 480x480 (3601 tokens), for batches of 48 and 64.  One model per shape (same weights),
the four arms alternating call by call in one process (CUDA events around each call, 3 warm-up rounds, 20 timed
rounds), then one profiled call per arm for the per-kind kernel times.  Prints one JSON line with the device name and
power limit (--out also writes it to a file).

The per-frame time of 480x640 over 480x480 should lie between the ratio of the token counts (1.33: GEMMs, MLP,
LayerNorms) and the ratio of their squares (1.78: attention)."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from dino_b200 import DINOSeg, _lib, synthetic  # noqa: E402
from features_timing import power_limit_w  # noqa: E402

WARMUP, STEPS = 3, 20


def run_batch(hws, batch, nb=3):
    lib = _lib.load()
    cfg = synthetic.make_config("vit_small", nb, 7)
    sd = synthetic.init_state_dict(cfg, 0, "reference_init")
    arms, models, tokens = {}, {}, {}
    for h, w in hws:
        m = DINOSeg(head="mlp", n_blocks=nb, n_classes=7, arch="vit_small")
        m.load_state_dict(sd, strict=True)
        m = m.to("cuda:0")
        g = torch.Generator().manual_seed(1)
        x = torch.randn(batch, 3, h, w, generator=g).cuda()
        m.infer(x, want_logprobs=False, want_lowres=True)          # handle, weights, resolution, workspace
        hd, ws, stream = m._handle, m._workspace, m._stream()
        n_tok = (h // 8) * (w // 8) + 1
        low = torch.empty((batch, h // 8, w // 8), dtype=torch.uint8, device="cuda")
        feats = torch.empty((1, batch, n_tok, cfg["embed_dim"]), dtype=torch.float32, device="cuda")
        tag = f"{h}x{w}"

        def forward(hd=hd, x=x, low=low, ws=ws, stream=stream):
            return lib.dinoseg_forward(hd, x.data_ptr(), batch, None, low.data_ptr(), None, ws.data_ptr(), ws.numel(),
                                       stream)

        def features(hd=hd, x=x, feats=feats, ws=ws, stream=stream):
            return lib.dinoseg_features(hd, x.data_ptr(), batch, 1, feats.data_ptr(), ws.data_ptr(), ws.numel(), stream)

        for kind, fn in (("forward", forward), ("features_n1", features)):
            arms[f"{kind}_{tag}"] = fn
            models[f"{kind}_{tag}"] = m
            tokens[f"{kind}_{tag}"] = n_tok
    launches = {}
    for name, fn in arms.items():
        assert fn() == 0, _lib.last_error(models[name]._handle)
        launches[name] = models[name].last_launch_count()
    times = {name: [] for name in arms}
    for step in range(WARMUP + STEPS):
        for name, fn in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            assert fn() == 0, _lib.last_error(models[name]._handle)
            e1.record()
            e1.synchronize()
            if step >= WARMUP:
                times[name].append(e0.elapsed_time(e1))
    out = {}
    for name, fn in arms.items():
        m = models[name]
        m.profile_enable(True)
        assert fn() == 0, _lib.last_error(m._handle)
        torch.cuda.synchronize()
        kinds = {k: [round(ms, 4), cnt] for k, (ms, cnt) in m.profile_read().items()}
        m.profile_enable(False)
        med = statistics.median(times[name])
        out[name] = {"frames_per_s": round(batch / (med / 1e3), 1),
                     "tokens_per_s": round(batch * tokens[name] / (med / 1e3), 0),
                     "ms_median": round(med, 4), "ms_min": round(min(times[name]), 4),
                     "ms_max": round(max(times[name]), 4), "launches": launches[name], "kernel_ms_by_kind": kinds}
    (sh, sw), (rh, rw) = hws
    ratios = {}
    for kind in ("forward", "features_n1"):
        sq, rect = out[f"{kind}_{sh}x{sw}"], out[f"{kind}_{rh}x{rw}"]
        ratios[kind] = round(rect["ms_median"] / sq["ms_median"], 4)
        ratios[kind + "_attention"] = round(rect["kernel_ms_by_kind"]["attention"][0] /
                                            sq["kernel_ms_by_kind"]["attention"][0], 4)
    n_sq, n_rect = (sh // 8) * (sw // 8) + 1, (rh // 8) * (rw // 8) + 1
    return {"arch": "vit_small", "n_blocks": nb, "batch": batch, "arms": out,
            "time_per_frame_ratio": ratios, "token_ratio": round(n_rect / n_sq, 4),
            "token_sq_ratio": round((n_rect / n_sq) ** 2, 4)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--hw", type=int, nargs=2, default=(480, 640), metavar=("H", "W"), help="non-square frame size")
    ap.add_argument("--square", type=int, default=480, help="side of the square frames it is compared with")
    ap.add_argument("--batches", type=int, nargs="+", default=(48, 64))
    ap.add_argument("--out", help="also write the JSON line to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rect_timing.py needs a GPU")
    hws = [(a.square, a.square), tuple(a.hw)]
    res = {"device": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(), "warmup": WARMUP, "steps": STEPS,
           "shapes": [run_batch(hws, b) for b in a.batches]}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Headline benchmark: frames/sec of the DINOSeg inference hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA library)
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on host cores

A "step" is one pass of the hot path (ViT-S/8 truncated to 3 blocks at 480 px -> MLP head ->
argmax -> 480x480 int64 label maps) over one batch of synthetic frames:
  N = 1 : 64 frames (BASELINE.json configs[1]);
  N > 1 : 512 frames sharded across the N GPUs, 256 / 128 / 64 per GPU (configs[2]; `scaling: "strong"`).
`--batch B` fixes the per-GPU batch instead (weak scaling), `--global-batch G` the global one.
Frames shard across ranks as independent replicas: no collective on the data path; NCCL is only
used for the barrier around the timed region and the max-over-ranks of the device time.
At N = 1 the line also carries `extra_configs`: BASELINE configs[3] (960 px, 16 frames) and configs[4]'s per-GPU
shape (ViT-B/8, 4 blocks, 480 px, 32 frames), measured in the same run (device-resident frames, CUDA events).

Output: ONE JSON line on rank 0 (see the keys below).  `value` is timed with CUDA events with the
frames already resident in HBM; `e2e` is the same metric through the public API
(`DINOSeg.predict_batch` on pinned HOST frames -> host label maps: H2D and D2H copies inside the
timed region); `roofline` describes the dominant kernel (attention, tensor-core bound);
`cpu_baseline` is the oracle (a port of the reference algorithm with the same ATen CPU kernels)
timed on this box's host cores on a bounded sample.

`--dump-outputs DIR` also writes the int64 label maps of the last timed step (what the caller of the timed path receives)
as DIR/labels.npy in float32 (labels_rank<r>.npy per rank on several GPUs), with the batch index of each frame in
DIR/labels_frames.npy: inputs and weights are seeded,
so two builds run with the same arguments can be compared map for map.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "frames/sec at 480px ViT-S/8 DINOSeg (n_blocks=3, MLP head, argmax + 480x480 label map)"
UNIT = "frames/s"
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}
DUMP_BUDGET = 64 << 20     # bytes written by --dump-outputs, all ranks together


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--batch", type=int, default=0, help="frames per GPU per step (0 = 64 on one GPU, 512 / N on N GPUs)")
    ap.add_argument("--global-batch", type=int, default=0, help="frames per step over all GPUs (overrides --batch)")
    ap.add_argument("--no-extra-configs", action="store_true", help="skip the 960 px / ViT-B side measurements (N = 1)")
    ap.add_argument("--res", type=int, default=480)
    ap.add_argument("--arch", default="vit_small")
    ap.add_argument("--n-blocks", type=int, default=3)
    ap.add_argument("--variant", default="reference_init", choices=["reference_init", "trained_like"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-sample-frames", type=int, default=0, help="0 = auto (bounded by ~20 s)")
    ap.add_argument("--kernels", action="store_true", help="add a per-kernel-kind breakdown (extra profiled pass)")
    ap.add_argument("--stall-limit", type=float, default=0.0,
                    help="seconds after which a run that has not finished is aborted with an error line instead of "
                         "hanging the box (0 = 300 s + 2 s per step)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the label maps of the last timed step to DIR/*.npy (float32; "
                         f"at most {DUMP_BUDGET >> 20} MB, a fixed sample of frames if the batch is larger)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    args.scaling = "weak"
    if args.global_batch > 0:
        if args.global_batch % world:
            ap.error(f"--global-batch {args.global_batch} is not a multiple of the {world} ranks")
        args.batch, args.scaling = args.global_batch // world, "strong"
    elif args.batch <= 0:
        # BASELINE.json: configs[1] = 64 frames on one GPU, configs[2] = 512 frames sharded across 2 / 4 / 8 GPUs
        args.batch = 64 if world == 1 else max(1, 512 // world)
        args.scaling = "weak" if world == 1 else "strong"
    return args


PHASE = ["start"]          # where the run is (reported by the stall watchdog)
STALL_HOOKS = []           # callables returning a diagnostic string


def arm_stall_watchdog(args):
    """A stalled run (GPU kernel that never returns, wedged collective, ...) must END: after the limit the process
    prints an error line and exits hard (os._exit tears the CUDA context down, which kills whatever is running)."""
    import threading
    limit = args.stall_limit if args.stall_limit > 0 else 300.0 + 2.0 * (args.steps + args.warmup)

    def fire():
        sys.stderr.write(f"bench.py: no result after {limit:.0f} s - aborting (phase: {PHASE[0]})\n")
        for hook in STALL_HOOKS:                    # what the GPU side says (registered once the model exists)
            try:
                sys.stderr.write(hook() + "\n")
            except Exception as e:                  # noqa: BLE001 - diagnostics must not mask the stall report
                sys.stderr.write(f"stall hook failed: {e}\n")
        try:                                        # where every thread of this process is stuck
            import faulthandler
            faulthandler.dump_traceback(file=sys.stderr, all_threads=True)
        except Exception:
            pass
        sys.stderr.flush()
        if int(os.environ.get("RANK", "0")) == 0:
            print(json.dumps({"error": f"stalled: no result after {limit:.0f} s", "impl": args.impl, "phase": PHASE[0]}),
                  flush=True)
        os._exit(3)

    t = threading.Timer(limit, fire)
    t.daemon = True
    t.start()
    return t


def kernel_options(model):
    """Opt-in library switches active in this run (DINOSEG_PAIR / DINOSEG_HOST_EXPAND or the C-ABI setters)."""
    from dino_b200 import _lib
    lib = _lib.load()
    pair = lib.dinoseg_get_pair_kernels(model._handle)
    return {"cta_pair_gemms": bool(pair & 1), "cta_pair_fused_mlp": bool(pair & 2),
            "host_label_expansion": lib.dinoseg_get_host_expand(model._handle) == 1}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured (MEASURED_PEAKS.json)"
    return dict(FALLBACK_PEAKS), "fallback (B200_PROFILING.md)"


def workload_name(args):
    a = {"vit_small": "ViT-S/8", "vit_base": "ViT-B/8"}[args.arch]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    shard = (f"batch {args.batch * world} synthetic frames sharded across {world} GPUs ({args.batch} per GPU)"
             if world > 1 else f"batch {args.batch} synthetic frames on 1 GPU")
    return f"{a} DINOSeg n_blocks={args.n_blocks}, {args.res}px, {shard}"


def ncu_attention_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the attention kernel, from the newest committed
    `ncu --set full` summary of the bench workload (profiles/r*_attn_ncu_full.csv, written by tools/ncu_summary.py)."""
    import csv
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_attn_ncu_full.csv")), reverse=True):
        try:
            with open(path) as f:
                rows = list(csv.DictReader(f))
        except OSError:
            continue
        for r in rows:
            if "attn_fwd_kernel" not in r.get("kernel", ""):
                continue
            try:
                rd = float(next(v for k, v in r.items() if k.startswith("dram_read")))
                wr = float(next(v for k, v in r.items() if k.startswith("dram_write")))
            except (StopIteration, ValueError):
                continue
            return (rd + wr) * 1e6, os.path.relpath(path, ROOT), r.get("block", "")
    return None, None, None


def dump_outputs(out_dir, name, labels, budget):
    """--dump-outputs: the int label maps [B, H, W] of the last timed step -> out_dir/<name>.npy as float32 (exact for class
    indices), and the batch index of every frame written -> out_dir/<name>_frames.npy (float64).  A batch that does not fit
    `budget` bytes is cut to a fixed, seeded sample of frames, the same in every run, so that two builds can be compared
    output for output."""
    import numpy as np
    import torch
    n = int(labels.shape[0])
    frame_bytes = labels[0].numel() * 4
    room = budget - 8 * n - 4096                     # the index array and two .npy headers
    keep = np.arange(n)
    if n * frame_bytes > room:
        keep = np.sort(np.random.default_rng(0).choice(n, max(1, room // frame_bytes), replace=False))
    out = labels[torch.from_numpy(keep).to(labels.device)].to(torch.float32).cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), out)
    np.save(os.path.join(out_dir, name + "_frames.npy"), keep.astype(np.float64))


# ------------------------------------------------------------------------------------------
# clocks during the timed region
# ------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()

    def summary(self, t0: float, t1: float):
        sm, mx, reasons, power = [], [], set(), []
        for t, line in self.rows:
            if t < t0 or t > t1 + 0.05:
                continue
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2])); power.append(float(parts[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power)}


# ------------------------------------------------------------------------------------------
# CPU legs (the oracle port of the reference algorithm) — the only place bench.py touches oracle/
# ------------------------------------------------------------------------------------------
def cpu_forward_timer(args, sd, cfg):
    import torch
    from oracle import dinoseg_oracle as O
    from dino_b200 import synthetic
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    g = args.res // 8

    def run(frames):
        lp = O.forward(sd, cfg, frames, frame_chunk=1)
        return O.labels_from_logprobs(lp, frames.shape[0], g)[1]

    return run, cores, synthetic


def cpu_baseline(args, sd, cfg, budget_s=20.0):
    """Oracle on host cores over a bounded sample of the same workload (frames of the same batch)."""
    run, cores, synthetic = cpu_forward_timer(args, sd, cfg)
    frames = synthetic.make_frames(min(args.batch, 8), args.res, seed=1)
    run(frames[:1])                                       # warm-up (thread pool, allocator)
    t0 = time.perf_counter()
    run(frames[:1])
    t1 = time.perf_counter() - t0
    n = args.cpu_sample_frames or int(max(1, min(frames.shape[0], budget_s // max(t1, 1e-3))))
    t0 = time.perf_counter()
    run(frames[:n])
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{n} of the batch's {args.batch} frames ({args.res}px, n_blocks={args.n_blocks}), fp32 torch CPU "
                      f"ops, {cores} threads, one frame at a time, forward+argmax+kron, after 1 warm-up frame"}


def run_reference_arm(args):
    """--impl reference: the reference algorithm (oracle port, same ATen CPU kernels as the reference's
    PyTorch path) on this box's host cores.  One step = a one-frame sample of the step's batch."""
    import torch
    from dino_b200 import synthetic
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cfg = synthetic.make_config(args.arch, args.n_blocks, 7)
    sd = synthetic.init_state_dict(cfg, 0, args.variant)
    run, cores, _ = cpu_forward_timer(args, sd, cfg)
    frames = synthetic.make_frames(1, args.res, seed=1)
    with torch.no_grad():
        for _ in range(max(1, args.warmup)):
            run(frames)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            labels = run(frames)
        dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, "labels", torch.from_numpy(labels), DUMP_BUDGET)
    fps = args.steps / dt
    sample = (f"1 frame per step out of the step's {args.batch}-frame batch ({args.res}px), fp32 torch CPU ops with "
              f"{cores} threads; frames are independent so frames/s does not depend on the sample size")
    out = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args), "sample": sample, "host_cores": cores},
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)
    return 0


# ------------------------------------------------------------------------------------------
# the B200 arm
# ------------------------------------------------------------------------------------------
def extra_configs(args, dev, peaks):
    """BASELINE.json configs[3] and configs[4] (per-GPU shape) on this GPU, in the same run: frames resident in HBM,
    CUDA events around `steps` passes after 3 warm-ups, events around every attention launch, clocks sampled during the
    timed region.  Parity of both shapes: tests/test_gpu_e2e.py::test_baseline_config_*."""
    import torch
    from dino_b200 import DINOSeg, synthetic
    from dino_b200.flops import attention_flops_per_launch, flops_per_frame
    peak_tf = float(peaks.get("bf16_tflops_sustained", FALLBACK_PEAKS["bf16_tflops_sustained"]))
    res_out = {}
    for key, arch, nb, res, batch in (("vit_s8_nb3_960px_b16", "vit_small", 3, 960, 16),
                                      ("vit_b8_nb4_480px_b32", "vit_base", 4, 480, 32)):
        cfg = synthetic.make_config(arch, nb, 7)
        m = DINOSeg(head="mlp", n_blocks=nb, n_classes=7, arch=arch)
        m.load_state_dict(synthetic.init_state_dict(cfg, 0, args.variant), strict=True)
        m = m.to(dev)
        m.set_resolution(res)
        x = synthetic.make_frames(batch, res, seed=3).to(dev)
        for _ in range(3):
            m.infer(x, want_logprobs=False, want_labels=True)
        torch.cuda.synchronize()
        steps = max(3, min(args.steps, 10))
        sampler = ClockSampler(dev.index or 0)
        sampler.start()
        time.sleep(0.25)
        m.profile_enable(True, kinds=("attention",))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record()
        for _ in range(steps):
            m.infer(x, want_logprobs=False, want_labels=True)
        e1.record()
        torch.cuda.synchronize()
        t1 = time.time()
        sampler.stop()
        ms = e0.elapsed_time(e1)
        att_ms, att_n = m.profile_read().get("attention", (0.0, 0))
        m.profile_enable(False)
        g = res // 8
        fl = attention_flops_per_launch(batch, g * g + 1, cfg["embed_dim"])
        fps = batch * steps / (ms / 1e3)
        step_tf = fps * flops_per_frame(cfg, res) / 1e12
        a = {"workload": f"{ {'vit_small': 'ViT-S/8', 'vit_base': 'ViT-B/8'}[arch]} DINOSeg n_blocks={nb}, {res}px, batch {batch} "
                         "synthetic frames on 1 GPU", "value": fps, "unit": UNIT, "steps": steps, "ms_per_step": ms / steps,
             "whole_step_tflops": step_tf, "whole_step_frac_of_sustained_peak": step_tf / peak_tf,
             "clocks": sampler.summary(t0, t1)}
        if att_n:
            ach = fl / (att_ms / att_n * 1e-3) / 1e12
            a["attention"] = {"achieved_tflops": ach, "frac_of_sustained_peak": ach / peak_tf, "avg_launch_ms": att_ms / att_n,
                              "tokens": g * g + 1, "heads": cfg["num_heads"], "share_of_step": att_ms / ms}
        res_out[key] = a
        del m, x
        torch.cuda.empty_cache()
    return res_out


def main():
    args = parse_args()
    arm_stall_watchdog(args)       # a run that does not finish ends with an error line and exit code 3; it is never retried
    if os.environ.get("DINOSEG_BENCH_TEST_STALL") == "1":     # test hook: behave like a run that never finishes
        time.sleep(1e9)
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    from dino_b200 import DINOSeg, dist as D, synthetic

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the DINOSeg hot path has no CPU fallback"}))
        return 1
    rank, local_rank, world = D.init()
    if world != args.gpus and rank == 0:
        print(f"[bench] note: --gpus {args.gpus} but WORLD_SIZE={world}; using {world}", file=sys.stderr)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    bound_cores = D.bind_to_gpu_cpus(local_rank) if world > 1 else 0   # NUMA-local host buffers for the e2e copies
    peaks, peaks_src = load_peaks()

    cfg = synthetic.make_config(args.arch, args.n_blocks, 7)
    sd = synthetic.init_state_dict(cfg, 0, args.variant)
    model = DINOSeg(head="mlp", n_blocks=args.n_blocks, n_classes=7, arch=args.arch)
    model.load_state_dict(sd, strict=True)
    model = model.to(dev)
    model.set_resolution(args.res)

    B, res, g = args.batch, args.res, args.res // 8
    # every rank owns its own shard of the global batch (different seeds per rank)
    frames_host = synthetic.make_frames(B, res, seed=1 + rank).pin_memory()
    frames = frames_host.to(dev, non_blocking=True)
    torch.cuda.synchronize()

    def step():
        return model.infer(frames, want_logprobs=False, want_labels=True)[2]

    def gpu_state():
        import ctypes as C
        from dino_b200 import _lib as _L
        lib = _L.load()
        kinds, slots, waiting = (C.c_int * 8)(), (C.c_int * 8)(), C.c_int(0)
        n = lib.dinoseg_debug_pending_kinds(model._handle, kinds, slots, 8, C.byref(waiting))
        running = [f"{lib.dinoseg_profile_kind_name(kinds[i]).decode()}#{slots[i]}" for i in range(max(n, 0))]
        smi = subprocess.run(["nvidia-smi", "--query-gpu=utilization.gpu,clocks.sm,power.draw,memory.used",
                              "--format=csv,noheader", "-i", str(local_rank)], capture_output=True, text=True, timeout=10).stdout.strip()
        hb = (C.c_int * 160)()
        nhb = lib.dinoseg_debug_heartbeat(hb, 160)
        live = {i: hb[i] for i in range(max(nhb, 0)) if hb[i] > 0}      # SM -> kernel code * 10 + stage (hb_mark)
        if os.environ.get("DINOSEG_BENCH_HB_WIDE") == "1":                # experimental builds: second half of the array
            hb2 = (C.c_int * 1024)()
            if lib.dinoseg_debug_heartbeat(hb2, 1024) > 0:
                live = {"stage": live, "alloc_returned": {i: hb2[512 + i] for i in live}}
        return (f"launches started and not finished: {running if n >= 0 else 'profiling off'}; queued behind them: "
                f"{waiting.value}; nvidia-smi: {smi}; tcgen05 CTAs still resident (sm: code*10+stage): {live}")

    STALL_HOOKS.append(gpu_state)
    PHASE[0] = "warm-up"

    for _ in range(max(3, args.warmup)):
        labels = step()
    torch.cuda.synchronize()
    launches_per_step = model.last_launch_count()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)

    # ---- timed region: device-resident inputs; events on the launching stream ----
    PHASE[0] = "timed region (device-resident frames)"
    # events around the dominant kernel only (DINOSEG_BENCH_ALL_EVENTS=1: around every launch, for stall diagnosis)
    model.profile_enable(True, kinds=None if os.environ.get("DINOSEG_BENCH_ALL_EVENTS") == "1" else ("attention",))
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    D.barrier()
    torch.cuda.synchronize()
    t_wall0 = time.time()
    ev0.record()
    for _ in range(args.steps):
        labels = step()
    ev1.record()
    torch.cuda.synchronize()
    D.barrier()
    t_wall1 = time.time()
    ms = ev0.elapsed_time(ev1)
    prof = model.profile_read()
    model.profile_enable(False)
    ms_max = D.max_over_ranks(ms)
    fps = world * B * args.steps / (ms_max / 1e3)

    # ---- end-to-end: pinned host frames -> public API -> host label maps ----
    # A caller that streams batches keeps two submissions in flight (DINOSeg.predict_batch_async / predict_wait): the
    # H2D copy of step k+1 overlaps the last kernels and the D2H copy of step k.  Every step still copies its own
    # frames from pinned host memory and delivers its own int64 label maps into (alternating) pinned host buffers.
    def e2e_loop(frames_in, resolution, outs):
        def run(n):
            prev = model.predict_batch_async(frames_in, resolution=resolution, output="labels", out=outs[0])
            for i in range(1, n):
                t = model.predict_batch_async(frames_in, resolution=resolution, output="labels", out=outs[i % 2])
                model.predict_wait(prev)
                prev = t
            return model.predict_wait(prev)
        run(3)
        D.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        last = run(args.steps)
        torch.cuda.synchronize()
        return D.max_over_ranks(time.perf_counter() - t0), last

    e2e = e2e_u8 = None
    PHASE[0] = "e2e (host frames, pipelined)"
    if os.environ.get("DINOSEG_BENCH_ALL_EVENTS") == "1":
        model.profile_enable(True)                 # stall diagnosis: events around every launch of the host path too
    if not args.no_e2e:
        from dino_b200 import _lib as _L
        side = 480 // g * g
        outs = [torch.empty((B, side, side), dtype=torch.int64).pin_memory() for _ in range(2)]
        dt_max, out = e2e_loop(frames_host, None, outs)
        # what crosses PCIe device -> host per step: the low-res maps when the library expands them into the int64
        # [480,480] maps with its host threads inside the same call (np.kron of the reference), else the int64 maps
        # replicated on the GPU (automatic choice by host cores per rank, dinoseg_set_host_expand)
        expand = _L.load().dinoseg_get_host_expand(model._handle) == 1
        d2h = int((B * g * g if expand else out.size * 8) * world)
        tail = ("low-res maps D2H, expanded to int64 label maps by the library's host threads"
                if expand else "int64 maps replicated on the GPU and copied out whole")
        e2e = {"value": world * B * args.steps / dt_max, "unit": UNIT,
               "h2d_bytes_per_step": int(frames_host.numel() * 4 * world),
               "d2h_bytes_per_step": d2h, "host_label_bytes_per_step": int(out.size * 8 * world),
               "api": "DINOSeg.predict_batch_async / predict_wait (pinned host fp32 frames -> int64 host label maps; "
                      "dinoseg_predict_host_submit / _wait: H2D + forward + D2H inside the timed region on the library's "
                      "copy-in / compute / copy-out streams, two steps in flight; " + tail + ")"}
        # ---- the same from RAW camera frames (uint8 640x480 RGB, as DINOSeg.predict receives them): resize + normalise
        # on the GPU as well; informational, the contract's `e2e` is the fp32 path above ----
        if res == 480:
            import numpy as np
            raw = torch.from_numpy(np.random.default_rng(7 + rank).integers(0, 256, (B, 480, 640, 3), dtype=np.uint8)).pin_memory()
            dt_max, _ = e2e_loop(raw, res, outs)
            e2e_u8 = {"value": world * B * args.steps / dt_max, "unit": UNIT, "h2d_bytes_per_step": int(raw.numel() * world),
                      "d2h_bytes_per_step": d2h, "host_label_bytes_per_step": int(outs[0].numel() * 8 * world),
                      "api": "DINOSeg.predict_batch_async(pinned host uint8 640x480 RGB frames) -> int64 host label maps "
                             "(cv2-exact bilinear resize + normalisation fused into the patch embed on the GPU)"}
    t_wall2 = time.time()
    clocks = None
    if rank == 0:
        sampler.stop()
        clocks = sampler.summary(t_wall0, t_wall1)

    # ---- per-kernel breakdown (optional, separate profiled pass; not part of `value`) ----
    kinds = None
    PHASE[0] = "per-kernel breakdown"
    if args.kernels:
        model.profile_enable(True)
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        span_ms, gap_ms = model.profile_gaps()        # first launch's start -> last launch's end, and the time between launches
        kinds = {k: {"ms_per_step": v[0] / 3, "launches_per_step": v[1] // 3} for k, v in model.profile_read().items()}
        kinds["(between launches, incl. the event records)"] = {"ms_per_step": gap_ms / 3, "launches_per_step": 0}
        kinds["(span of the 3 profiled steps / 3)"] = {"ms_per_step": span_ms / 3, "launches_per_step": 0}
        model.profile_enable(False)

    # ---- roofline of the dominant kernel: fused attention (tensor-core bound) ----
    from dino_b200.flops import attention_flops_per_launch, flops_per_frame
    att_ms, att_n = prof.get("attention", (0.0, 0))
    N = g * g + 1
    f_launch = attention_flops_per_launch(B, N, cfg["embed_dim"])
    peak_tf = float(peaks.get("bf16_tflops_sustained", FALLBACK_PEAKS["bf16_tflops_sustained"]))
    peak_burst = float(peaks.get("bf16_tflops", FALLBACK_PEAKS["bf16_tflops"]))
    roofline = None
    if att_n:
        ach = f_launch / (att_ms / att_n * 1e-3) / 1e12
        traffic, traffic_src, traffic_block = (ncu_attention_traffic() if (B, res, args.arch) == (64, 480, "vit_small")
                                               else (None, None, None))
        roofline = {"kernel": "attn_fwd_kernel<6, true> (fused QK^T -> softmax without row maxima -> PV, tcgen05/TMEM) "
                              "+ the empty launch of its range-redo twin, timed together", "bound": "tensor",
                    "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                    # the kernel is timed inside a step that keeps the GPU under load, hence `peak` = the SUSTAINED cuBLAS
                    # figure; the fraction of the burst figure (a kernel timed alone on a cool GPU) is given beside it
                    "peak_burst": peak_burst, "frac_of_burst": ach / peak_burst,
                    # dram__bytes_read.sum + dram__bytes_write.sum per launch, parsed from the committed ncu --set full
                    # summary of this workload (algorithmic: 531 MB of q/k/v read once + 177 MB of output)
                    "traffic": traffic, "traffic_unit": "bytes per launch", "traffic_source": traffic_src,
                    "traffic_block_dim": traffic_block,
                    "peak_source": peaks_src + ", sustained figure (kernel timed inside a long step)",
                    "flops_per_launch": f_launch, "launches_timed": att_n, "avg_launch_ms": att_ms / att_n,
                    "share_of_step": att_ms / ms}
    F = flops_per_frame(cfg, res)
    step_tf = fps / world * F / 1e12

    out = {
        "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": workload_name(args), "global_batch": world * B, "weights": f"random init ({args.variant})",
                   "parallelism": f"replicas x{world} (frames sharded, no collective)", "host_cores_bound_per_rank": bound_cores,
                   "l2": "inputs+workspace per step (>1.5 GB) exceed the 126 MB L2; no explicit flush",
                   "arithmetic": "bf16 tensor-core operands, fp32 accumulate / residual stream / LN / softmax / GELU",
                   "kernel_options": kernel_options(model)},
        "clocks": clocks, "e2e": e2e, "e2e_u8": e2e_u8, "gpu_launches": int(launches_per_step * args.steps),
        "roofline": roofline,
        "whole_step": {"gflop_per_frame": F / 1e9, "achieved_tflops_per_gpu": step_tf, "frac_of_peak": step_tf / peak_tf,
                       "frac_of_burst": step_tf / peak_burst},
    }
    if kinds is not None:
        out["kernels"] = kinds
    if args.dump_outputs:                                          # `labels` is still the last timed step's result
        dump_outputs(args.dump_outputs, "labels" if world == 1 else f"labels_rank{rank}", labels, DUMP_BUDGET // world)
    if world == 1 and not args.no_extra_configs and (args.arch, args.res, args.n_blocks) == ("vit_small", 480, 3):
        del model, frames, labels                                  # free the workspace of the headline workload
        torch.cuda.empty_cache()
        out["extra_configs"] = extra_configs(args, dev, peaks)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:      # N = 1 only (bench contract)
        out["cpu_baseline"] = cpu_baseline(args, sd, cfg)
    if rank == 0:
        print(json.dumps(out), flush=True)
    D.barrier()
    D.shutdown()
    return 0


if __name__ == "__main__":
    sys.exit(main())

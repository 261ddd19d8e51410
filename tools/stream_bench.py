#!/usr/bin/env python
"""Cost of many-stream video mode on one GPU: capture_graph(B) (fused_forward: batch parse, no smoothing) against
capture_graph(B, streams=StreamStates(B)) (stream_forward: per-frame parse + per-stream OneEuro smoothing), replays
of the two graphs alternated on the same device, then -- in a separate profiled run -- the device times of the
parse_* and one_euro_kernel kernels.

    python tools/stream_bench.py [--batch 256] [--steps 60] [--warmup 5] [--out profiles/stream_bench_b256.json]

Prints one JSON object (and writes it to --out): ms/step from CUDA events per arm (median and spread over the
timed steps), frames/s, the difference, the kernel table, and the card name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
for p in (os.path.join(ROOT, "arbitrary-hands-3d-reconstruction_b200"), ROOT):
    sys.path.insert(0, p)
os.environ.setdefault("ACR_B200_SYNTHETIC_MANO", "1")


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.steps < 50:
        raise SystemExit("--steps must be >= 50")
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("stream_bench needs a CUDA device")
    from acr.config import args as cfg
    from acr.main import ACR
    from acr_b200 import ops
    from acr_b200.synth import load_bn_calibration, make_synthetic_mano, synth_state_dict
    cfg().return_maps = False
    B = a.batch
    app = ACR(state_dict=synth_state_dict(0, bn_stats=load_bn_calibration(0)),
              mano_assets={"left": make_synthetic_mano("left"), "right": make_synthetic_mano("right")})
    g = torch.Generator().manual_seed(0)
    frames = torch.randint(0, 256, (B, 512, 512, 3), generator=g, dtype=torch.uint8).cuda()
    offs = torch.tensor([[512., 512, 0, 0, 0, 0, 0, 0, 0, 0]]).repeat(B, 1).cuda()
    states = ops.StreamStates(B, "cuda")
    plain = app.capture_graph(B)
    streams = app.capture_graph(B, streams=states)
    ids = torch.arange(B, dtype=torch.int32).cuda()     # device ids: the copy into the graph's buffer stays on-device
    arms = {"fused_forward": lambda: plain(frames, offs), "stream_forward": lambda: streams(frames, offs, ids)}
    for _ in range(a.warmup):
        for f in arms.values():
            f()
    torch.cuda.synchronize()
    ms = {k: [] for k in arms}
    for _ in range(a.steps):
        for k, f in arms.items():          # alternate the arms step by step
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            e1.synchronize()
            ms[k].append(e0.elapsed_time(e1))
    res = {"card": card(), "batch": B, "steps": a.steps, "warmup": a.warmup, "arms": {}}
    for k, v in ms.items():
        v = np.array(v)
        res["arms"][k] = {"ms_per_step_median": round(float(np.median(v)), 3), "ms_p10": round(float(np.percentile(v, 10)), 3),
                          "ms_p90": round(float(np.percentile(v, 90)), 3),
                          "frames_per_s": round(B / float(np.median(v)) * 1e3, 1)}
    d = np.array(ms["stream_forward"]) - np.array(ms["fused_forward"])
    res["diff_ms_median"] = round(float(np.median(d)), 3)
    res["diff_ms_p10_p90"] = [round(float(np.percentile(d, 10)), 3), round(float(np.percentile(d, 90)), 3)]

    # kernel times, separate profiled run (eager launches so that every kernel is attributed)
    from torch.profiler import ProfilerActivity, profile
    for _ in range(2):
        app.fused_forward(frames, offs)
        app.stream_forward(frames, offs, states, ids)
    torch.cuda.synchronize()
    n_prof = 10
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n_prof):
            app.fused_forward(frames, offs)
            app.stream_forward(frames, offs, states, ids)
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.key_averages():
        name = ev.key
        if "parse_" in name or "one_euro" in name:
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = ev.cuda_time_total
            kern[name] = {"calls": ev.count, "us_per_call": round(t / max(ev.count, 1), 2)}
    res["kernels"] = kern
    res["kernel_note"] = (f"{n_prof} eager fused_forward + {n_prof} eager stream_forward at B={B} under torch.profiler; "
                          "parse_scan runs in fused_forward only, parse_slot and one_euro_kernel in stream_forward only")
    print(json.dumps(res, indent=1), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

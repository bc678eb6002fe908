"""High-resolution forward timings of the full model (random weights, images only): ms per forward under CUDA-graph
replay, global-attention ms per launch (CUDA events around each launch of an eager pass, ovg_runtime_time_attention) with
its share of the B200 data-sheet bf16 dense peak, peak device memory, and the card name / power limit read in the same
process.  One JSON line per config.

    python tools/hires_bench.py [--steps 10] [--warmup 3] [--configs wide1036,sq1036,sq2044,cfg2] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# name -> (views, H, W); cfg2 (8 x 518^2) is the control at the size bench.py measures
CONFIGS = {
    "wide1036": (8, 784, 1036),      # what --target_size 1036 makes of 4:3 images
    "sq1036": (8, 1036, 1036),
    "sq2044": (2, 2044, 2044),       # the edge of the supported envelope (146 x 146 patches)
    "cfg2": (8, 518, 518),
}
BF16_DENSE_PEAK_TFLOPS = 2250.0      # NVIDIA HGX B200 data sheet, one GPU, dense, at 1 000 W (not a measured rate)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]], capture_output=True, text=True)
    return q.stdout.strip() or q.stderr.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--configs", default=",".join(CONFIGS))
    ap.add_argument("--out", help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    from omnivggt_official_b200 import OmniVGGT, _lib
    from oracle.synth import make_inputs
    assert torch.cuda.is_available(), "hires_bench measures on a GPU"
    dev = torch.device("cuda", 0)
    with torch.device(dev):
        m = OmniVGGT(init_seed=None)
    m.randomize_(0).eval()
    lib = _lib.lib()
    gpu = card()
    for name in args.configs.split(","):
        S, H, W = CONFIGS[name]
        m._graphs = {}
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats(dev)
        images = make_inputs(1, S, H, W, seed=1)["images"].to(dev)
        m.use_cuda_graph = True
        for _ in range(max(args.warmup, 3)):          # the third call of a signature captures the graph later calls replay
            m(images=images)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            m(images=images)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.steps
        # eager pass: single launches inside a replayed graph cannot be bracketed by events
        m.use_cuda_graph = False
        m(images=images)
        torch.cuda.synchronize()
        lib.ovg_runtime_time_attention(1)
        m(images=images)
        torch.cuda.synchronize()
        buf = (ctypes.c_float * 4096)()
        n = lib.ovg_runtime_attention_times(ctypes.cast(buf, ctypes.c_void_p), 4096)
        lib.ovg_runtime_time_attention(0)
        att = [buf[i] for i in range(max(n, 0))]
        att_ms = sum(att) / max(len(att), 1)
        P = (H // 14) * (W // 14)
        L = S * (P + 5)
        flops = 4.0 * L * L * 1024                     # QK^T + PV, 16 heads x 64, per launch
        tflops = flops / (att_ms * 1e-3) / 1e12
        line = {"config": name, "views": S, "H": H, "W": W, "rope_positions": max(H, W) // 14 + 1, "tokens_per_frame": P + 5,
                "global_seq": L, "ms_per_forward": round(ms, 2), "steps": args.steps, "launch": "CUDA graph replay",
                "global_attention": {"launches": len(att), "ms_per_launch": round(att_ms, 4), "tflops": round(tflops, 1),
                                     "share_of_bf16_datasheet_peak": round(tflops / BF16_DENSE_PEAK_TFLOPS, 3),
                                     "timed_in": "separate eager forward"},
                "share_of_forward_in_global_attention": round(sum(att) / ms, 3),
                "peak_memory_gib": round(torch.cuda.max_memory_allocated(dev) / 2 ** 30, 2),
                "gpu": gpu, "weights": "random, full architecture", "inputs": "images only"}
        print(json.dumps(line), flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(json.dumps(line) + "\n")
        del images


if __name__ == "__main__":
    main()

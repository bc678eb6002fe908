#!/usr/bin/env python
"""Benchmark of the OmniVGGT hot path (BASELINE.json metric: view-sets/sec, N-view 518^2 batches).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config cfg1..cfg5] [--dump-outputs DIR]

One "step" = the full OmniVGGT.forward over this rank's share of the workload.  Workloads (BASELINE.json configs[0..4]):
  cfg1  1 scene x 4 views @ 518^2, images only
  cfg2  1 scene x 8 views @ 518^2, images only                      <- default, the N = 1 headline
  cfg3  1 scene x 8 views @ 518^2, depth + camera aux on all views
  cfg4  32 scenes x 8 views @ 518^2, images only, scenes sharded over the ranks (strong scaling), micro-batches of scenes
  cfg5  1 scene x 24 views @ 518^2, partial depth_gt_index / camera_gt_index
cfg1/2/3/5 under torchrun: weak scaling, one independent view-set per rank per step; weights broadcast once from rank 0 (NCCL).
Prints ONE JSON line on rank 0 (DESIGN.md section "Measurement" defines the fields).
--dump-outputs DIR writes rank 0's predictions of the last timed step to DIR (see dump_outputs); inputs and weights are
seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

IMG = 518
T_TOK = (IMG // 14) ** 2 + 5
CONFIGS = {
    "cfg1": dict(S=4, scenes=1, depth_idx=[], cam_idx=[], scaling="weak",
                 desc="cfg1: 1 scene x 4 views @ 518x518, images-only, per GPU per step (BASELINE.json configs[0])"),
    "cfg2": dict(S=8, scenes=1, depth_idx=[], cam_idx=[], scaling="weak",
                 desc="cfg2: 1 scene x 8 views @ 518x518, images-only, per GPU per step (BASELINE.json configs[1])"),
    "cfg3": dict(S=8, scenes=1, depth_idx=list(range(8)), cam_idx=list(range(8)), scaling="weak",
                 desc="cfg3: 1 scene x 8 views @ 518x518, depth + camera aux on all 8 views, per GPU per step (BASELINE.json configs[2])"),
    "cfg4": dict(S=8, scenes=32, depth_idx=[], cam_idx=[], scaling="strong",
                 desc="cfg4: 32 scenes x 8 views @ 518x518, images-only, scenes sharded over the ranks (BASELINE.json configs[3])"),
    "cfg5": dict(S=24, scenes=1, depth_idx=[0, 3, 4, 9, 15, 22], cam_idx=[0, 1, 2, 7, 11, 12, 20, 23], scaling="weak",
                 desc="cfg5: 1 scene x 24 views @ 518x518, partial depth / camera aux, per GPU per step (BASELINE.json configs[4])"),
}
OUT_KEYS = ("pose_enc", "depth", "depth_conf", "world_points", "world_points_conf")
DUMP_BYTES = 60_000_000          # payload cap of --dump-outputs (with the .npy headers the files stay under 64 MB)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1393.7), d.get("hbm_gbs", 6489.9), "measured (MEASURED_PEAKS.json, sustained bf16)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


def synth_inputs(B, S, seed):
    """Synthetic inputs shaped like the tuple reference visual_util.py:835-841 feeds the model (SURVEY.md section 8d recipe):
    images U[0,1), random world->camera poses, pinhole intrinsics, depth 0.5 + 4 U[0,1) with ~20% invalid pixels."""
    import torch
    g = torch.Generator().manual_seed(seed)
    images = torch.rand(B, S, 3, IMG, IMG, generator=g)
    q, r = torch.linalg.qr(torch.randn(B * S, 3, 3, generator=g))
    q = q * torch.sign(torch.diagonal(r, dim1=-2, dim2=-1))[:, None, :]
    q[:, :, 0] = q[:, :, 0] * torch.linalg.det(q)[:, None]
    extr = torch.cat([q.reshape(B, S, 3, 3), torch.randn(B, S, 3, 1, generator=g)], -1)
    intr = torch.zeros(B, S, 3, 3)
    intr[..., 0, 0] = intr[..., 1, 1] = 500.0
    intr[..., 0, 2] = intr[..., 1, 2] = IMG / 2
    intr[..., 2, 2] = 1.0
    mask = (torch.rand(B, S, IMG, IMG, generator=g) > 0.2).float()
    depth = (0.5 + 4.0 * torch.rand(B, S, IMG, IMG, 1, generator=g)) * mask[..., None]
    return dict(images=images, extrinsics=extr, intrinsics=intr, depth=depth, mask=mask)


def dump_outputs(outs, directory, limit=DUMP_BYTES):
    """Write what one step returned to its caller as ``directory/<name>.npy`` (float32).  ``outs`` holds the output dict of
    every forward call of the step; the calls are concatenated along the scene axis, ``pose_enc_list`` is written as
    ``pose_enc_list.<i>``.  ``images`` (the caller's own input, handed back unchanged) and non-tensor entries are skipped.
    If the arrays exceed ``limit`` bytes together, the smallest are kept whole and every array larger than its share of
    what is left is replaced by a sample of its flattened elements: the sorted indices drawn without replacement by
    ``numpy.random.default_rng(zlib.crc32(name))``, so that the same arguments give the same sample on every run."""
    import numpy as np
    import torch
    arrays = {}
    for k, v in outs[0].items():
        if k == "pose_enc_list":
            for i in range(len(v)):
                arrays[f"{k}.{i}"] = torch.cat([o[k][i] for o in outs]).float().cpu().numpy()
        elif torch.is_tensor(v) and k != "images":
            arrays[k] = torch.cat([o[k] for o in outs]).float().cpu().numpy()
    os.makedirs(directory, exist_ok=True)
    left = limit
    for n, (name, a) in enumerate(sorted(arrays.items(), key=lambda kv: kv[1].nbytes)):
        share = left // (len(arrays) - n)
        if a.nbytes > share:
            idx = np.random.default_rng(zlib.crc32(name.encode())).choice(a.size, share // a.itemsize, replace=False)
            a = a.reshape(-1)[np.sort(idx)]
        left -= a.nbytes
        np.save(os.path.join(directory, name + ".npy"), a)


class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.p = index, None

    def __enter__(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None
        time.sleep(0.25)
        return self

    def __exit__(self, *a):
        self.out = ""
        if self.p is not None:
            time.sleep(0.15)
            self.p.terminate()
            try:
                self.out = self.p.communicate(timeout=5)[0]
            except Exception:
                self.p.kill()

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx = max(mx, float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v == "Active":
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ reference arm (CPU)
def run_reference(args, rank, world):
    """The reference's own CPU implementation of the path on the host cores, rank 0 only: the UNMODIFIED reference
    ``OmniVGGT.forward`` (omnivggt/models/omnivggt.py:20-68, fp32, torch.no_grad) imported from oracle/_ref (packed there
    by oracle/vendor_ref.py in the build container) and run on the arm's config -- one warm-up forward, then whole timed
    forwards until --steps or the time budget is reached (at least 2).  ``steps`` in the line = forwards actually timed.
    Without oracle/_ref the arm falls back to the oracle-port unit sampler, labelled ``kind: "port"``."""
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1 to its workers; this arm must use every host core it can get, so the variables
    # are dropped BEFORE torch / MKL / OpenMP initialise
    for var in ("OMP_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ.pop(var, None)
    import torch
    cfg = CONFIGS[args.config]
    S = cfg["S"]
    budget = float(os.environ.get("OVG_REF_BUDGET_S", "200"))
    kind, sample, secs = "reference", "", []
    try:
        from oracle.vendor_ref import import_reference_zip
        Ref = import_reference_zip()
    except Exception:
        Ref = None
    if Ref is not None:
        t0 = time.perf_counter()
        model = Ref().eval()                       # stock random init of the full architecture (no checkpoint offline)
        build_s = time.perf_counter() - t0
        inp = synth_inputs(1, S, seed=1)
        kw = dict(images=inp["images"], extrinsics=inp["extrinsics"], intrinsics=inp["intrinsics"], depth=inp["depth"],
                  mask=inp["mask"], depth_gt_index=list(cfg["depth_idx"]), camera_gt_index=list(cfg["cam_idx"]))
        warm = 1 if args.warmup > 0 else 0
        with torch.no_grad():
            for _ in range(warm):
                model(**kw)
            t_begin = time.perf_counter()
            while len(secs) < max(args.steps, 1):
                t0 = time.perf_counter()
                model(**kw)
                secs.append(time.perf_counter() - t0)
                if len(secs) >= 2 and time.perf_counter() - t_begin + secs[-1] > budget:
                    break
        per_scene = statistics.median(secs)
        sample = (f"unmodified reference OmniVGGT.forward (oracle/_ref), fp32 CPU, 1 scene x {S} views @ {IMG}x{IMG}, "
                  f"{warm} warm-up + {len(secs)} timed whole forwards (model build {build_s:.0f} s outside the timed region)")
    else:
        from oracle import cpu_baseline as cb
        kind, warm = "port", 1 if args.warmup else 0
        for _ in range(warm):
            cb.sample(S)
        t_begin = time.perf_counter()
        for _ in range(args.steps):
            secs.append(cb.sample(S)[0])
            if time.perf_counter() - t_begin > budget:
                break
        per_scene = statistics.median(secs)
        sample = "FALLBACK (oracle/_ref missing): " + cb.SAMPLE_DESC
    # cfg4: the CPU processes the 32 scenes one after the other -> one step = 32 forwards; a step sample is one scene x 32
    step_s = per_scene * cfg["scenes"]
    val = cfg["scenes"] / step_s
    line = {"impl": "reference", "metric": "view_sets_per_sec", "value": val, "unit": "view-sets/s", "n_gpus": args.gpus,
            "steps": len(secs), "warmup": warm, "ms_per_step": step_s * 1e3, "higher_is_better": True,
            "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["desc"], "device": "host CPU", "name": args.config},
            "cpu_baseline": {"value": val, "unit": "view-sets/s", "cores": torch.get_num_threads(), "kind": kind,
                             "sample": sample},
            "e2e": {"value": val, "unit": "view-sets/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU library baseline
def gpu_torch_baseline(model, inputs, cfg, dev, ours):
    """The real competitor (SURVEY.md section 8d): the UNMODIFIED reference on the same B200 through the library kernels
    PyTorch dispatches to (cuBLAS, cuDNN, SDPA), fp32 as inference.py runs it and under torch.autocast(bf16), with OUR
    weights loaded (same 1 505 keys).  Runs after the product arm's timed regions.  Also reports output deviations:
    ours vs reference fp32, and reference-bf16-autocast vs reference fp32 (the yardstick of SURVEY.md section 8d)."""
    import torch
    from oracle.vendor_ref import import_reference_zip
    Ref = import_reference_zip()
    with torch.device(dev):
        ref = Ref()
    ref.load_state_dict(model.state_dict(), strict=True)
    ref = ref.to(dev).eval()
    kw = dict(images=inputs["images"], extrinsics=inputs["extrinsics"], intrinsics=inputs["intrinsics"],
              depth=inputs["depth"], mask=inputs["mask"], depth_gt_index=list(cfg["depth_idx"]),
              camera_gt_index=list(cfg["cam_idx"]))

    def timed(ctx, n=3):
        with torch.no_grad(), ctx():
            out = ref(**kw)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                out = ref(**kw)
            e1.record()
            torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n, out

    import contextlib
    ms32, _ = timed(contextlib.nullcontext)
    ms16, out16 = timed(lambda: torch.autocast("cuda", dtype=torch.bfloat16))
    # the deviations are taken against true fp32: PyTorch's default lets cuDNN run the heads' fp32 convolutions in TF32
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    with torch.no_grad():
        out32 = ref(**kw)
    torch.backends.cudnn.allow_tf32 = tf32

    def rel(a, b):
        return float((a.float() - b.float()).norm() / b.float().norm().clamp(min=1e-12))

    res = {"what": "unmodified reference OmniVGGT.forward on this GPU (library kernels), our weights, same inputs",
           "fp32_ms": ms32, "bf16_autocast_ms": ms16,
           "fp32_view_sets_per_s": 1e3 / ms32, "bf16_autocast_view_sets_per_s": 1e3 / ms16,
           "rel_l2_ours_vs_ref_fp32": {k: rel(ours[k], out32[k]) for k in OUT_KEYS},
           "rel_l2_ref_bf16_autocast_vs_ref_fp32": {k: rel(out16[k], out32[k]) for k in OUT_KEYS}}
    del ref, out32, out16
    torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------------------------------ product arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS))
    ap.add_argument("--scene-batch", type=int, default=4, help="cfg4: scenes per forward call")
    ap.add_argument("--cp", action="store_true", help="context parallelism: ONE scene per step, its views sharded over the ranks")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-torch-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the predictions of the last timed step as DIR/<name>.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the predictions of --impl b200")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        return run_reference(args, rank, world)
    args.warmup = max(args.warmup, 3)
    cfg = CONFIGS[args.config]

    import torch
    import torch.distributed as dist
    from omnivggt_official_b200 import OmniVGGT, _lib
    from omnivggt_official_b200.dist import broadcast_weights, max_over_ranks, shard_scenes

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    S = cfg["S"]
    with torch.device(dev):
        model = OmniVGGT(init_seed=None)
    model.randomize_(seed=0 if rank == 0 else 1000 + rank)     # non-zero ranks are overwritten by the broadcast
    bcast_bytes = 0
    if world > 1:
        bcast_bytes = broadcast_weights(model, src=0)
    model.eval()
    eng = model.engine()
    lib = _lib.lib()

    # ---- this rank's share of the workload: `calls` forward calls of `Bm` scenes each per step
    if args.cp:
        # one scene per step for the whole job: every rank gets the full (replicated) inputs and computes its views
        assert cfg["scenes"] == 1 and S % world == 0, "--cp shards the views of a single-scene config over the ranks"
        model.enable_context_parallel()
        Bm, calls, total_scenes = 1, 1, 1
    elif cfg["scaling"] == "strong":
        mine = shard_scenes(cfg["scenes"], rank, world)
        Bm = max(1, min(args.scene_batch, len(mine)))
        while len(mine) % Bm:
            Bm -= 1
        calls = len(mine) // Bm
        total_scenes = cfg["scenes"]
    else:
        Bm, calls = 1, 1
        total_scenes = world
    need_d, need_c = len(cfg["depth_idx"]) > 0, len(cfg["cam_idx"]) > 0
    in_keys = ["images"] + (["depth", "mask"] if need_d else []) + (["extrinsics", "intrinsics"] if need_c else [])
    host_in = [{k: v.pin_memory() for k, v in synth_inputs(Bm, S, seed=1 + (0 if args.cp else rank * 64) + c).items() if k in in_keys}
               for c in range(calls)]
    dev_in = [{k: v.to(dev) for k, v in h.items()} for h in host_in]
    idx_kw = dict(depth_gt_index=list(cfg["depth_idx"]), camera_gt_index=list(cfg["cam_idx"]))
    host_out = [None] * calls
    step_out = []

    def step_resident():
        step_out[:] = [model(**dev_in[c], **idx_kw) for c in range(calls)]

    from omnivggt_official_b200.pipeline import StreamingPipeline
    pipe = StreamingPipeline(model, slots=2, out_keys=OUT_KEYS)
    pending = []

    def step_e2e():
        """One step end to end through the public streaming API: every step copies its own inputs from pinned host memory and
        reads its own predictions back to pinned host memory; the copies of neighbouring steps overlap this step's forward on
        separate streams (pipeline.py).  The previous step's result is collected here, the last one in e2e_drain()."""
        for c in range(calls):
            pending.append(pipe.submit(host_in[c], **idx_kw))
            if len(pending) > 1:
                host_out[c] = pipe.result(pending.pop(0))

    def e2e_drain():
        while pending:
            host_out[0] = pipe.result(pending.pop(0))
        pipe.drain()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        return max_over_ranks(ms, dev) if world > 1 else ms

    for _ in range(args.warmup):        # (the third call of a shape captures the CUDA graph that later calls replay)
        step_resident()
    with ClockSampler(local) as cs:
        total_ms = timed(step_resident, args.steps)
    clocks = cs.summary()
    if args.dump_outputs and rank == 0:
        dump_outputs(step_out, args.dump_outputs)
    ms_step = total_ms / args.steps
    value = total_scenes * 1e3 / ms_step

    for _ in range(args.warmup):
        step_e2e()
    e2e_drain()

    def e2e_run():
        for _ in range(args.steps):
            step_e2e()
        e2e_drain()            # the last step's device->host read is inside the timed region

    e2e_ms = timed(e2e_run, 1) / args.steps

    # Kernel-level pass: the product path replays a CUDA graph, inside which single launches cannot be bracketed by
    # events or counted by the library, so the same K steps are run once more with eager launches to time the 24
    # global-attention launches per forward and to count libovg launches per step.
    graph_mode = model.use_cuda_graph
    model.use_cuda_graph = False
    step_resident()
    if os.environ.get("OVG_BENCH_PROFILE_RANGE"):      # `ncu --profile-from-start off`: exactly one step of this command
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        step_resident()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
    lib.ovg_runtime_time_attention(1)          # the runtime brackets every global-attention launch with CUDA events
    l0 = lib.ovg_launch_count()
    timed(step_resident, args.steps)
    launches = (lib.ovg_launch_count() - l0) // args.steps
    import ctypes
    buf = (ctypes.c_float * 8192)()
    n_att = lib.ovg_runtime_attention_times(ctypes.cast(buf, ctypes.c_void_p), 8192)
    lib.ovg_runtime_time_attention(0)
    att_ms = [buf[i] for i in range(max(n_att, 0))]
    model.use_cuda_graph = graph_mode
    h2d = sum(t.numel() * t.element_size() for h in host_in for t in h.values())
    d2h = sum(t.numel() * t.element_size() for h in host_out for t in h.values())

    # ---- roofline of the dominant kernel: global attention (24 launches / forward), timed live with CUDA events
    peak_tf, peak_hbm, peak_src = measured_peaks()
    L = S * T_TOK
    att_flops = 4.0 * Bm * L * L * 1024               # SURVEY.md section 8d: 4 L^2 C per scene and launch (QK^T + PV, 16 heads x 64)
    if args.cp:
        att_flops /= world                            # a rank's own queries (L / world rows) against all L keys
    att_avg = sum(att_ms) / max(len(att_ms), 1)
    achieved = att_flops / (att_avg * 1e-3) / 1e12
    traffic = None
    tp = os.path.join(ROOT, "profiles", "attn_traffic.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get(f"S{S}") if Bm == 1 else None
    roofline = {"kernel": "ovg::attn1_kernel (global attention)", "bound": "tensor", "achieved": achieved, "peak": peak_tf,
                "unit": "TFLOP/s", "frac": achieved / peak_tf, "traffic": traffic, "peak_source": peak_src,
                "launches_timed": len(att_ms), "avg_launch_ms": att_avg,
                "share_of_step": sum(att_ms) / args.steps / ms_step,
                "timed_in": "separate eager pass of the same K steps (launches inside the replayed CUDA graph cannot be bracketed)"}

    line = {"metric": "view_sets_per_sec", "value": value, "unit": "view-sets/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong" if args.cp else cfg["scaling"],
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "dtype_note": "aggregator / DINOv2 / camera head: bf16 operands, fp32 accumulation and residual stream; DPT heads: "
                          + model.dpt_dtype + " operands and maps, fp32 accumulation",
            "config": {"workload": cfg["desc"], "name": args.config, "views": S,
                       "scenes_per_step_all_ranks": total_scenes, "scenes_per_forward_call": Bm, "forward_calls_per_step_per_rank": calls,
                       "depth_gt_index": cfg["depth_idx"], "camera_gt_index": cfg["cam_idx"],
                       "parallelism": (f"cp{world}: views of one scene sharded over the ranks; K/V rows exchanged by peer stores from the QKV "
                                       f"epilogue + flag barrier, no collective on the data path" if args.cp else
                                       f"dp{world} (scene-sharded, NCCL weight broadcast {bcast_bytes} B at start-up)"),
                       "weights": "random-init, full architecture (1217.5 M params)",
                       "l2": "no flush needed: each step streams >2 GB of weights+activations, far beyond the 126 MB L2",
                       "dino": "frozen DINOv2 patchifier on the libovg kernels",
                       "launch": "CUDA graph replay" if model.use_cuda_graph else "eager (C++ runtime sequences)"},
            "clocks": clocks,
            "e2e": {"value": total_scenes * 1e3 / e2e_ms, "unit": "view-sets/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms},
            "gpu_launches": int(launches), "roofline": roofline}

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import cpu_baseline as cb
        import torch as _t
        est, parts = cb.sample(S)
        line["cpu_baseline"] = {"value": 1.0 / est, "unit": "view-sets/s", "cores": _t.get_num_threads(), "kind": "port",
                                "sample": cb.SAMPLE_DESC, "seconds_per_view_set": est}
    if rank == 0 and world == 1 and not args.no_gpu_torch_baseline and Bm == 1 and not args.cp:
        try:
            ours = model(**dev_in[0], **idx_kw)
            full_in = {k: v.to(dev) for k, v in synth_inputs(1, S, seed=1).items()}
            line["gpu_torch_baseline"] = gpu_torch_baseline(model, full_in, cfg, dev, ours)
        except Exception as ex:   # a baseline leg must never cost the product line
            import traceback
            line["gpu_torch_baseline"] = {"unavailable": repr(ex)[:300], "where": traceback.format_exc()[-600:]}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

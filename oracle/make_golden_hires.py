"""High-resolution parity pins: the UNMODIFIED reference ``OmniVGGT`` (full architecture, reference
omnivggt/models/omnivggt.py:10-68) above 882 px per side, where the 2-D RoPE grid has more than 64 positions per axis
(build container only; TEST INFRASTRUCTURE).

    python oracle/make_golden_hires.py            # CPU fp32; minutes per case

Cases:
  hires_wide_s2   1 scene x 2 views @ 784 x 1036, images only (what ``--target_size 1036`` makes of a 4:3 image; 75 positions)
  hires_aux_s3    1 scene x 3 views @ 1036 x 1036, depth_gt_index [0, 2], camera_gt_index [0, 1]

Weights are oracle/synth.make_state_dict(schema, seed 0) over tests/golden/full.schema.json (checked against the reference
module's own state dict; the file is not rewritten).  Dense outputs are stored on a lattice of every 14th row / column
(offset 7), fp32.  Writes tests/golden/hires_*.safetensors and tests/golden/hires_index.json.
"""
from __future__ import annotations

import json
import os
import sys
import time

import torch
from safetensors.torch import save_file

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle.ref_shims import import_reference  # noqa: E402
from oracle.synth import make_inputs, make_state_dict  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(HERE), "tests", "golden")
STRIDE = 14

# name -> (S, H, W, depth_gt_index, camera_gt_index, input seed)
CASES = {
    "hires_wide_s2": (2, 784, 1036, [], [], 21),
    "hires_aux_s3": (3, 1036, 1036, [0, 2], [0, 1], 22),
}


def lattice(t: torch.Tensor) -> torch.Tensor:
    """[B,S,H,W,...] -> every STRIDE-th pixel (offset STRIDE // 2)."""
    o = STRIDE // 2
    return t[:, :, o::STRIDE, o::STRIDE].contiguous().clone()


def main():
    import_reference()
    from omnivggt.models.omnivggt import OmniVGGT as RefOmniVGGT
    torch.set_num_threads(os.cpu_count() or 8)
    only = set(sys.argv[1:])
    m = RefOmniVGGT().eval()
    schema = json.load(open(os.path.join(GOLDEN, "full.schema.json")))["schema"]
    assert schema == {k: list(t.shape) for k, t in m.state_dict().items()}, "reference schema differs from full.schema.json"
    sd = make_state_dict(schema, seed=0)
    m.load_state_dict(sd, strict=True)
    del sd
    path = os.path.join(GOLDEN, "hires_index.json")
    index = json.load(open(path)) if os.path.exists(path) else {}
    for name, (S, H, W, didx, cidx, seed) in CASES.items():
        if only and name not in only:
            continue
        inp = make_inputs(1, S, H, W, seed=seed)
        t0 = time.time()
        with torch.no_grad():
            out = m(images=inp["images"], extrinsics=inp["extrinsics"], intrinsics=inp["intrinsics"], depth=inp["depth"],
                    mask=inp["mask"], depth_gt_index=list(didx), camera_gt_index=list(cidx))
        dt = time.time() - t0
        store = {"pose_enc": out["pose_enc"].contiguous().clone()}
        for i, p in enumerate(out["pose_enc_list"]):
            store[f"pose_enc_list.{i}"] = p.contiguous().clone()
        for k in ("depth", "depth_conf", "world_points", "world_points_conf"):
            store[k] = lattice(out[k].float())
        save_file(store, os.path.join(GOLDEN, f"{name}.safetensors"))
        stats = {k: [float(v.abs().mean()), float(v.abs().max())] for k, v in store.items() if "list" not in k}
        index[name] = dict(S=S, H=H, W=W, depth_gt_index=didx, camera_gt_index=cidx, input_seed=seed, weight_seed=0,
                           stride=STRIDE, cpu_forward_s=round(dt, 1), cpu_threads=torch.get_num_threads(), stats=stats)
        print(name, f"{dt:.0f} s", stats, flush=True)
        with open(path, "w") as f:
            json.dump(index, f, indent=1, sort_keys=True)


if __name__ == "__main__":
    main()

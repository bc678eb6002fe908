"""Images above 882 px per side (GPU): the QKV epilogue with more RoPE positions than its shared-memory table holds (cos / sin
read from the global tables), parity with the unmodified reference at 784 x 1036 and 1036 x 1036, the full model at the edge
of the supported envelope (2 044 x 2 044), and the GPU loader at ``target_size=1036``.

Tolerances are the ones of the 518 x 518 pins (tests/test_model_gpu.py): rel-L2 1e-2 per output with the default fp16 DPT
heads, pose_enc max-abs 5e-2; kernel level 6e-3 (bf16 outputs)."""
import json
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from safetensors.torch import load_file

from conftest import GOLDEN
from oracle import postprocess_oracle as POST
from oracle import preprocess_oracle as PO
from oracle.synth import make_inputs
from test_kernels_gpu import _rope_ref, randn, rel
from test_model_gpu import KEYS, TOL_FP16_HEADS, full_model, model
from test_preprocess import _read_folder

pytestmark = pytest.mark.gpu
BF16 = torch.bfloat16
HIRES_INDEX = json.load(open(os.path.join(GOLDEN, "hires_index.json")))
GOLD_PRE = json.load(open(os.path.join(GOLDEN, "preprocess_hires.json")))


def _qkv(C, frames, hp, wp, ntok, bn, cos, sin, seed=1):
    """One QKV epilogue launch into sentinel-guarded outputs; returns (q, k, v, inputs, guard buffers)."""
    from omnivggt_official_b200 import ops
    heads, T = C // 64, hp * wp + 5
    M = frames * T
    a = randn(M, C, seed=seed, dtype=BF16)
    w = randn(3 * C, C, scale=C ** -0.5, seed=seed + 1, dtype=BF16)
    bias = randn(3 * C, scale=0.1, seed=seed + 2)
    ln = (1 + 0.1 * randn(64, seed=seed + 3), 0.1 * randn(64, seed=seed + 4), 1 + 0.1 * randn(64, seed=seed + 5), 0.1 * randn(64, seed=seed + 6))
    nb = M // ntok
    guard = 4096
    bufs = [torch.full((guard + nb * heads * ntok * 64 + guard,), 7.0, device="cuda", dtype=BF16) for _ in range(3)]
    q, k, v = (b[guard:-guard].view(nb, heads, ntok, 64) for b in bufs)
    for t in (q, k, v):
        t.zero_()
    ops.qkv_proj(a, w, bias, *ln, q, k, v, ntok=ntok, T=T, nspecial=5, wp=wp, rope_cos=cos, rope_sin=sin, block_n=bn)
    return q, k, v, (a, w, bias, ln), bufs, guard


@pytest.mark.parametrize("bn", [0, 128, 512])
@pytest.mark.parametrize("C,hp,wp", [(1024, 56, 74), (256, 146, 146)])
def test_qkv_epilogue_large_rope_grid(C, hp, wp, bn):
    """QKV linear + q/k LayerNorm + 2-D RoPE with 75 / 147 positions per axis against the fp32 formulas
    (layers/attention.py:52-58, layers/rope.py:154-188), frame-wise and global token layouts."""
    from omnivggt_official_b200 import ops
    frames, S = 2, 2
    heads, T = C // 64, hp * wp + 5
    cos, sin = ops.rope_tables(max(hp, wp) + 1, "cuda")
    assert cos.shape[0] > 64
    for ntok in (T, S * T):
        q, k, v, (a, w, bias, (qn_w, qn_b, kn_w, kn_b)), bufs, guard = _qkv(C, frames, hp, wp, ntok, bn, cos, sin)
        nb = frames * T // ntok
        qkv = (a.float() @ w.float().t() + bias).reshape(nb, ntok, 3, heads, 64).permute(2, 0, 3, 1, 4)
        yy, xx = torch.meshgrid(torch.arange(hp, device="cuda"), torch.arange(wp, device="cuda"), indexing="ij")
        pos = torch.cat([torch.zeros(5, 2, device="cuda", dtype=torch.long), torch.stack([yy.reshape(-1), xx.reshape(-1)], -1) + 1])
        pos = pos[None].expand(frames, -1, -1).reshape(nb, ntok, 2)
        qr = _rope_ref(F.layer_norm(qkv[0], (64,), qn_w, qn_b, 1e-5), pos) * (math.log2(math.e) / 8.0)
        kr = _rope_ref(F.layer_norm(qkv[1], (64,), kn_w, kn_b, 1e-5), pos)
        torch.cuda.synchronize()
        errs = (rel(q, qr), rel(k, kr), rel(v, qkv[2]))
        assert max(errs) < 6e-3, errs
        for b in bufs:
            assert (b[:guard] == 7.0).all() and (b[-guard:] == 7.0).all()
        del q, k, v, qkv, qr, kr, bufs
        torch.cuda.empty_cache()


@pytest.mark.parametrize("bn", [0, 128, 512])
def test_qkv_epilogue_global_table_path_equals_smem_path(bn):
    """The same 37 x 37 grid once with a 100-row table (cos / sin from global memory) and once with its first 38 rows (the
    shared-memory table): the two epilogues read the same fp32 entries and must agree bit for bit."""
    from omnivggt_official_b200 import ops
    cos, sin = ops.rope_tables(100, "cuda")
    small = (cos[:38].contiguous(), sin[:38].contiguous())
    T = 37 * 37 + 5
    for ntok in (T, 2 * T):
        big = _qkv(1024, 2, 37, 37, ntok, bn, cos, sin)[:3]
        ref = _qkv(1024, 2, 37, 37, ntok, bn, *small)[:3]
        torch.cuda.synchronize()
        for name, x, y in zip("qkv", big, ref):
            assert torch.equal(x, y), (name, ntok, bn)


@pytest.mark.parametrize("case", sorted(HIRES_INDEX))
def test_hires_matches_reference_golden(case):
    """The full model against outputs of the UNMODIFIED reference forward (CPU fp32, oracle/make_golden_hires.py) at sizes
    with more than 64 RoPE positions per axis; dense outputs on the stored lattice (every 14th pixel, offset 7)."""
    meta = HIRES_INDEX[case]
    m = full_model()
    if m.dpt_dtype != "fp16":
        m.dpt_dtype = "fp16"
        m._invalidate()
    st, o = meta["stride"], meta["stride"] // 2
    inp = {k: v.cuda() for k, v in make_inputs(1, meta["S"], meta["H"], meta["W"], seed=meta["input_seed"]).items()}
    out = m(depth_gt_index=meta["depth_gt_index"], camera_gt_index=meta["camera_gt_index"], **inp)
    torch.cuda.synchronize()
    ref = load_file(os.path.join(GOLDEN, f"{case}.safetensors"))
    got = {"pose_enc": out["pose_enc"]}
    for k in KEYS[1:]:
        assert torch.isfinite(out[k]).all(), k
        got[k] = out[k][:, :, o::st, o::st]
    errs = {k: rel(got[k].cpu(), ref[k]) for k in KEYS}
    errs["pose_enc_maxabs"] = (out["pose_enc"].cpu() - ref["pose_enc"]).abs().max().item()
    for i in range(4):
        errs[f"pose_enc_list.{i}"] = rel(out["pose_enc_list"][i].cpu(), ref[f"pose_enc_list.{i}"])
    line = f"{case} H={meta['H']} W={meta['W']} S={meta['S']} " + json.dumps({k: round(v, 5) for k, v in errs.items()})
    print(line)
    for k in KEYS:
        assert got[k].shape == ref[k].shape, k
        assert errs[k] < TOL_FP16_HEADS, (k, errs)
    assert errs["pose_enc_maxabs"] < 5e-2, errs


def test_envelope_edge_2044_properties():
    """2 044 x 2 044 (146 x 146 patches, 21 321 tokens per frame), 2 views, partial aux: output contract, finiteness,
    run-to-run and eager-vs-graph-replay bit identity, and the aux inputs reach the predictions."""
    m = full_model()
    S, H, W = 2, 2044, 2044
    didx, cidx = [0], [1]
    inp = {k: v.cuda() for k, v in make_inputs(1, S, H, W, seed=6).items()}
    graph = m.use_cuda_graph
    m.use_cuda_graph = True
    try:
        outs = [{k: v.clone() for k, v in m(depth_gt_index=didx, camera_gt_index=cidx, **inp).items() if k in KEYS}
                for _ in range(4)]     # call 3 captures, call 4 replays
        torch.cuda.synchronize()
        a = outs[0]
        assert a["depth"].shape == (1, S, H, W, 1) and a["world_points"].shape == (1, S, H, W, 3)
        assert a["depth_conf"].shape == (1, S, H, W) and a["pose_enc"].shape == (1, S, 9)
        for k in KEYS:
            assert torch.isfinite(a[k]).all(), k
            for o in outs[1:]:
                assert torch.equal(o[k], a[k]), k
        assert (a["depth"] > 0).all() and (a["depth_conf"] >= 1).all() and (a["world_points_conf"] >= 1).all()
        b = m(depth_gt_index=[], camera_gt_index=[], **inp)
        assert rel(b["depth"], a["depth"]) > 1e-4 and rel(b["pose_enc"], a["pose_enc"]) > 1e-4
    finally:
        m.use_cuda_graph = graph
        m._graphs = {}
        torch.cuda.empty_cache()


@pytest.mark.parametrize("name", sorted(GOLD_PRE.keys() - {"_versions", "_target_size"}))
def test_gpu_loader_at_1036_matches_oracle_bit_for_bit(name, tmp_path):
    from omnivggt_official_b200 import preprocess as PP
    from oracle.synth_folder import make_folder
    ts = GOLD_PRE["_target_size"]
    d = make_folder(str(tmp_path), name, seed=0)
    imgs, cams, deps, tr = _read_folder(d)
    ref = PO.load_views(imgs, cams, [x.T if t else x for x, t in zip(deps, tr)], target_size=ts)
    out = PP.load_images_and_cameras(d["images"], d["cameras"], d["depths"], target_size=ts)
    torch.cuda.synchronize()
    assert list(out[0].shape) == GOLD_PRE[name]["images_shape"]
    assert out[5] == ref[5] and out[6] == ref[6]
    assert torch.equal(out[0].cpu(), torch.from_numpy(ref[0]))
    assert torch.equal(out[3].cpu(), torch.from_numpy(ref[3])) and torch.equal(out[4].cpu(), torch.from_numpy(ref[4]))
    assert np.allclose(out[1].cpu().numpy(), ref[1], atol=2e-6) and np.allclose(out[2].cpu().numpy(), ref[2], rtol=1e-6, atol=1e-4)


def test_loader_forward_postprocess_at_1036(tmp_path):
    """loader (target_size=1036) -> forward -> postprocess on the 4:3 folder: 784 x 1036 views, 75 RoPE positions."""
    from omnivggt_official_b200 import preprocess as PP
    from oracle.synth_folder import make_folder
    d = make_folder(str(tmp_path), "wide", seed=0)
    images, extr, intr, dep, mask, didx, cidx = PP.load_images_and_cameras(d["images"], d["cameras"], d["depths"], target_size=1036)
    assert tuple(images.shape[-2:]) == (784, 1036)
    m = model("mini_conv")
    pred = m.postprocess(m(images=images, extrinsics=extr, intrinsics=intr, depth=dep, mask=mask, depth_gt_index=didx,
                           camera_gt_index=cidx), conf_percent=50.0)
    torch.cuda.synchronize()
    S = images.shape[0]
    assert pred["depth"].shape == (1, S, 784, 1036, 1) and pred["extrinsic"].shape == (1, S, 3, 4)
    assert pred["world_points_from_depth"].shape == (1, S, 784, 1036, 3) and pred["conf_mask"].shape == pred["depth_conf"].shape
    for k in ("depth", "depth_conf", "world_points"):
        assert torch.isfinite(pred[k]).all(), k
    # camera decoding at the 784 x 1036 image size (the reduced random-weight model may predict a degenerate field of view,
    # which the reference decodes to non-finite focals as well: compared NaN-aware)
    ext, intr = POST.pose_encoding_to_extri_intri(pred["pose_enc"].cpu().numpy(), 784, 1036)
    assert np.allclose(pred["extrinsic"].cpu().numpy(), ext, rtol=1e-4, atol=1e-5, equal_nan=True)
    assert np.allclose(pred["intrinsic"].cpu().numpy(), intr, rtol=1e-4, atol=1e-3, equal_nan=True)

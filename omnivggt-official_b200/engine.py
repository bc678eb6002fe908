"""Hot-path engine: weight repacking into kernel layouts and device-buffer ownership for the libovg RUNTIME handles.
The launch sequences of the aggregator (reference models/omnivggt_aggregator.py:130-305), of the frozen DINOv2 patchifier
(layers/vision_transformer.py:214-271) and of the DPT heads (heads/dpt_head.py:128-304) live in C++
(csrc/runtime.inc: ovg_aggregator_forward / ovg_dino_forward / ovg_dpt_forward); this file packs the checkpoint tensors
once, describes them to the library (ovg_*_desc), owns workspaces / outputs and makes one C call per component."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, fields
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib as L
from . import ops
from .torch_parts import pack_injection, uv_posembed_separable, uv_posembed_table

BF16, F32 = torch.bfloat16, torch.float32


def _bf(t: torch.Tensor) -> torch.Tensor:
    return t.detach().to(BF16).contiguous()


def _f32(t: torch.Tensor) -> torch.Tensor:
    return t.detach().to(F32).contiguous()


def _half(t: torch.Tensor, dtype) -> torch.Tensor:
    """16-bit kernel operand: bf16, or fp16 clamped to the finite range."""
    if dtype == torch.float16:
        return t.detach().float().clamp(-65504.0, 65504.0).to(dtype).contiguous()
    return t.detach().to(dtype).contiguous()


def _conv3x3_w(w: torch.Tensor, dtype=BF16) -> torch.Tensor:
    """[Cout, Cin, 3, 3] -> [Cout, 9*Cin], K order (tap = ky*3+kx, cin): matches the row-shifted tap GEMM."""
    return _half(w.permute(0, 2, 3, 1).reshape(w.shape[0], -1), dtype)


@dataclass
class BlockPack:
    ln1_w: torch.Tensor; ln1_b: torch.Tensor; w_qkv: torch.Tensor; b_qkv: torch.Tensor
    qn_w: torch.Tensor; qn_b: torch.Tensor; kn_w: torch.Tensor; kn_b: torch.Tensor
    w_proj: torch.Tensor; b_proj: torch.Tensor; g1: torch.Tensor
    ln2_w: torch.Tensor; ln2_b: torch.Tensor; w_fc1: torch.Tensor; b_fc1: torch.Tensor
    w_fc2: torch.Tensor; b_fc2: torch.Tensor; g2: torch.Tensor


def pack_block(bp) -> BlockPack:
    a = bp.attn
    qk = hasattr(a, "q_norm")       # aggregator blocks have q/k LayerNorm; DINOv2 blocks do not
    return BlockPack(_f32(bp.norm1.weight), _f32(bp.norm1.bias), _bf(a.qkv.weight), _f32(a.qkv.bias),
                     _f32(a.q_norm.weight) if qk else None, _f32(a.q_norm.bias) if qk else None,
                     _f32(a.k_norm.weight) if qk else None, _f32(a.k_norm.bias) if qk else None,
                     _bf(a.proj.weight), _f32(a.proj.bias), _f32(bp.ls1.gamma),
                     _f32(bp.norm2.weight), _f32(bp.norm2.bias), _bf(bp.mlp.fc1.weight), _f32(bp.mlp.fc1.bias),
                     _bf(bp.mlp.fc2.weight), _f32(bp.mlp.fc2.bias), _f32(bp.ls2.gamma))


def block_struct(bp: BlockPack) -> L.BlockWeights:
    w = L.BlockWeights()
    for f in fields(bp):
        setattr(w, f.name, L.ptr(getattr(bp, f.name)))
    return w


def _block_array(packs: Sequence[BlockPack]):
    arr = (L.BlockWeights * len(packs))()
    for i, bp in enumerate(packs):
        arr[i] = block_struct(bp)
    return arr


class DPTPack:
    """Kernel-layout weights of one DPT head.  The shared LayerNorm affine (heads/dpt_head.py:66,:227) is folded
    into the 1x1 projections: W (g*xhat + b) + c = (W*g) xhat + (W b + c).  ``dtype``: torch.float16 (default: the reference keeps
    its heads in fp32 even under autocast, models/omnivggt.py:45; IEEE half has the 11-bit significand of the TF32 convolutions PyTorch
    runs them with on a GPU, at the bf16 tensor-core rate) or torch.bfloat16 (wider exponent range, 8-bit significand)."""

    def __init__(self, hp, dtype=torch.float16):
        self.dtype = dtype
        _bf = lambda t: _half(t, dtype)                                          # noqa: E731  (all 16-bit operands of this head)
        _c3 = lambda w: _conv3x3_w(w, dtype)                                     # noqa: E731
        g, b = hp.norm.weight.detach().float(), hp.norm.bias.detach().float()
        self.proj_w, self.proj_b = [], []
        for pr in hp.projects:
            w = pr.weight.detach().float().flatten(1)            # [oc, 2C]
            self.proj_w.append(_bf(w * g[None]))
            self.proj_b.append(_f32(w @ b + pr.bias.detach().float()))
        self.oc = [w.shape[0] for w in self.proj_w]
        r0, r1, r3 = hp.resize_layers["0"], hp.resize_layers["1"], hp.resize_layers["3"]
        # ConvTranspose2d weight [Cin, Cout, k, k] -> rows (ky, kx, cout), cols cin
        self.up_w = [_bf(r.weight.detach().permute(2, 3, 1, 0).reshape(-1, r.weight.shape[0])) for r in (r0, r1)]
        self.up_b = [_f32(r0.bias), _f32(r1.bias)]
        self.down_w, self.down_b = _c3(r3.weight.detach()), _f32(r3.bias)
        s = hp.scratch
        self.rn_w = [_c3(getattr(s, f"layer{i + 1}_rn").weight.detach()) for i in range(4)]
        self.feat = self.rn_w[0].shape[0]
        self.fus = []
        for name in ("refinenet1", "refinenet2", "refinenet3", "refinenet4"):
            f = getattr(s, name)
            d = {"oc_w": _bf(f.out_conv.weight.detach().flatten(1)), "oc_b": _f32(f.out_conv.bias)}
            for u in ("resConfUnit1", "resConfUnit2"):
                if hasattr(f, u):
                    ru = getattr(f, u)
                    d[u] = (_c3(ru.conv1.weight.detach()), _f32(ru.conv1.bias),
                            _c3(ru.conv2.weight.detach()), _f32(ru.conv2.bias))
            self.fus.append(d)
        self.oc1_w, self.oc1_b = _c3(s.output_conv1.weight.detach()), _f32(s.output_conv1.bias)
        self.oc2_w, self.oc2_b = _c3(s.output_conv2["0"].weight.detach()), _f32(s.output_conv2["0"].bias)
        self.w2, self.b2 = _f32(s.output_conv2["2"].weight.detach().flatten(1)), _f32(s.output_conv2["2"].bias)
        self.outc = self.w2.shape[0]

    def desc(self, C2: int, patch: int) -> L.DptDesc:
        d = L.DptDesc()
        d.C2, d.feat, d.patch, d.outc = C2, self.feat, patch, self.outc
        for l in range(4):
            d.oc[l] = self.oc[l]
            d.proj_w[l], d.proj_b[l] = L.ptr(self.proj_w[l]), L.ptr(self.proj_b[l])
            d.rn_w[l] = L.ptr(self.rn_w[l])
            fu = self.fus[l]
            for k, u in enumerate(("resConfUnit1", "resConfUnit2")):
                dst = d.fus[l].rcu1 if k == 0 else d.fus[l].rcu2
                for j in range(4):
                    dst[j] = L.ptr(fu[u][j]) if u in fu else None
            d.fus[l].oc_w, d.fus[l].oc_b = L.ptr(fu["oc_w"]), L.ptr(fu["oc_b"])
        for l in range(2):
            d.up_w[l], d.up_b[l] = L.ptr(self.up_w[l]), L.ptr(self.up_b[l])
        d.down_w, d.down_b = L.ptr(self.down_w), L.ptr(self.down_b)
        d.oc1_w, d.oc1_b, d.oc2_w, d.oc2_b = L.ptr(self.oc1_w), L.ptr(self.oc1_b), L.ptr(self.oc2_w), L.ptr(self.oc2_b)
        d.w2, d.b2 = L.ptr(self.w2), L.ptr(self.b2)
        d.f16 = int(self.dtype == torch.float16)
        return d


class Workspace:
    """Named device buffers, reused across calls (stable addresses keep the TMA descriptor cache hot)."""

    def __init__(self, device):
        self.device = device
        self.bufs: Dict[str, torch.Tensor] = {}
        self.version = 0          # bumped on every (re)allocation: captured CUDA graphs hold raw pointers

    def get(self, name: str, shape: Sequence[int], dtype=BF16, zero: bool = False) -> torch.Tensor:
        n = 1
        for s in shape:
            n *= int(s)
        key = name
        buf = self.bufs.get(key)
        if buf is None or buf.dtype != dtype or buf.numel() < n:
            buf = torch.empty(max(n, 1), device=self.device, dtype=dtype)
            self.bufs[key] = buf
            self.version += 1
        v = buf[:n].view(*shape)
        if zero:
            v.zero_()
        return v


class Engine:
    def __init__(self, model):
        self.m = model
        self.device = next(model.parameters()).device
        ag = model.aggregator
        self.C = ag.camera_token.shape[-1]
        self.R = ag.register_token.shape[2]
        self.depth = len(ag.frame_blocks)
        self.heads = self.C // 64
        if self.C % 64:
            raise ValueError(f"embed_dim {self.C}: the attention / QKV kernels are built for head_dim 64 (embed_dim % 64 == 0)")
        self.patch = model.patch_size
        lib = L.lib()
        # ---- packed weights (kept alive here: the runtime handles only hold their device pointers)
        self.frame = [pack_block(b) for b in ag.frame_blocks]
        self.glob = [pack_block(b) for b in ag.global_blocks]
        self.cam_tok = _f32(ag.camera_token.reshape(2, self.C))
        self.reg_tok = _f32(ag.register_token.reshape(2, self.R, self.C))
        self.placeholder = _f32(ag.depth_placeholder.reshape(self.C))
        dw = ag.depth_patch_embed.proj.weight.detach()
        self.depth_w = _bf(dw.flatten(1))                         # [C, 2*patch*patch], K order (ch, ky, kx)
        self.depth_b = _f32(ag.depth_patch_embed.proj.bias)
        self.ones_c = torch.ones(self.C, device=self.device, dtype=F32)
        self.inj_pack = pack_injection(ag)
        self.keep = tuple(model.dpt_layers)
        self._handles = []
        d = L.AggregatorDesc()
        d.C, d.registers, d.depth, d.patch = self.C, self.R, self.depth, self.patch
        self._fb, self._gb = _block_array(self.frame), _block_array(self.glob)
        d.frame_blocks, d.global_blocks = self._fb, self._gb
        d.cam_tok, d.reg_tok, d.placeholder = L.ptr(self.cam_tok), L.ptr(self.reg_tok), L.ptr(self.placeholder)
        d.depth_w, d.depth_b, d.ones_c = L.ptr(self.depth_w), L.ptr(self.depth_b), L.ptr(self.ones_c)
        for i in range(4):
            d.keep_layers[i] = self.keep[i]
        self.h_agg = C.c_void_p()
        L.check(lib.ovg_aggregator_create(C.byref(d), C.byref(self.h_agg)))
        self._handles.append((lib.ovg_aggregator_destroy, self.h_agg))
        # frozen DINOv2 patchifier on the same kernels (SURVEY.md section 8f rank 1): reference
        # layers/vision_transformer.py:214-271 -- blocks without RoPE / q-k norm, LayerNorm eps 1e-6, LayerScale gammas
        self.dino = None
        pe = ag.patch_embed
        if hasattr(pe, "blocks") and getattr(model, "dino_backend", "ovg") == "ovg":
            if self.C // pe.heads != 64:
                raise ValueError(f"DINOv2 patchifier with head_dim {self.C // pe.heads}: libovg attention needs head_dim 64 "
                                 "(use dino_backend='torch' for other widths)")
            w = pe.patch_embed.proj.weight.detach().flatten(1)                       # [C, 3*p*p]
            kpad = (w.shape[1] + 7) // 8 * 8
            wpad = torch.zeros(w.shape[0], kpad, device=self.device, dtype=BF16)
            wpad[:, :w.shape[1]] = w.to(BF16)
            self.dino = dict(blocks=[pack_block(b) for b in pe.blocks], w=wpad, b=_f32(pe.patch_embed.proj.bias),
                             norm_w=_f32(pe.norm.weight), norm_b=_f32(pe.norm.bias), nreg=pe.register_tokens.shape[1], kpad=kpad)
            dd = L.DinoDesc()
            dd.C, dd.registers, dd.depth, dd.patch, dd.kpad = self.C, self.dino["nreg"], len(pe.blocks), self.patch, kpad
            self._db = _block_array(self.dino["blocks"])
            dd.blocks = self._db
            dd.w_patch, dd.b_patch = L.ptr(wpad), L.ptr(self.dino["b"])
            dd.norm_w, dd.norm_b, dd.ones_c = L.ptr(self.dino["norm_w"]), L.ptr(self.dino["norm_b"]), L.ptr(self.ones_c)
            self.h_dino = C.c_void_p()
            L.check(lib.ovg_dino_create(C.byref(dd), C.byref(self.h_dino)))
            self._handles.append((lib.ovg_dino_destroy, self.h_dino))
        dpt_dtype = {"fp16": torch.float16, "bf16": BF16}[getattr(model, "dpt_dtype", "fp16")]
        self.dpt_packs = {name: DPTPack(getattr(model, name), dpt_dtype) for name in ("depth_head", "point_head")
                          if getattr(model, name, None) is not None}
        self.h_dpt = {}
        for name, pk in self.dpt_packs.items():
            h = C.c_void_p()
            desc = pk.desc(2 * self.C, self.patch)
            L.check(lib.ovg_dpt_create(C.byref(desc), C.byref(h)))
            self.h_dpt[name] = h
            self._handles.append((lib.ovg_dpt_destroy, h))
        # camera head (reference heads/camera_head.py:83-154) on the same GEMM kernels + small fp32 kernels
        self.h_cam = None
        cp = getattr(model, "camera_head", None)
        if cp is not None and getattr(model, "camera_backend", "ovg") == "ovg":
            D = cp.token_norm.weight.shape[0]
            self.cam = dict(trunk=[pack_block(b) for b in cp.trunk], tn_w=_f32(cp.token_norm.weight), tn_b=_f32(cp.token_norm.bias),
                            rn_w=_f32(cp.trunk_norm.weight), rn_b=_f32(cp.trunk_norm.bias),
                            empty=_f32(cp.empty_pose_tokens.reshape(9)), ew=_f32(cp.embed_pose.weight), eb=_f32(cp.embed_pose.bias),
                            mw=_bf(cp.poseLN_modulation["1"].weight), mb=_f32(cp.poseLN_modulation["1"].bias),
                            f1w=_bf(cp.pose_branch.fc1.weight), f1b=_f32(cp.pose_branch.fc1.bias),
                            f2w=_f32(cp.pose_branch.fc2.weight), f2b=_f32(cp.pose_branch.fc2.bias), D=D)
            cd = L.CameraDesc()
            cd.D, cd.heads, cd.trunk_depth = D, cp.heads, len(cp.trunk)
            self._cb = _block_array(self.cam["trunk"])
            cd.trunk = self._cb
            c = self.cam
            cd.token_norm_w, cd.token_norm_b, cd.trunk_norm_w, cd.trunk_norm_b = L.ptr(c["tn_w"]), L.ptr(c["tn_b"]), L.ptr(c["rn_w"]), L.ptr(c["rn_b"])
            cd.empty_pose, cd.embed_w, cd.embed_b = L.ptr(c["empty"]), L.ptr(c["ew"]), L.ptr(c["eb"])
            cd.mod_w, cd.mod_b, cd.fc1_w, cd.fc1_b = L.ptr(c["mw"]), L.ptr(c["mb"]), L.ptr(c["f1w"]), L.ptr(c["f1b"])
            cd.fc2_w, cd.fc2_b = L.ptr(c["f2w"]), L.ptr(c["f2b"])
            self.h_cam = C.c_void_p()
            L.check(lib.ovg_camera_create(C.byref(cd), C.byref(self.h_cam)))
            self._handles.append((lib.ovg_camera_destroy, self.h_cam))
        self.ws = Workspace(self.device)
        self._idx_cache: Dict[tuple, torch.Tensor] = {}   # small device index tensors (no per-call H2D copies)
        self._rope: Dict[int, Tuple[torch.Tensor, torch.Tensor]] = {}
        self._tables: Dict[tuple, torch.Tensor] = {}

    def __del__(self):
        for destroy, h in getattr(self, "_handles", []):
            try:
                destroy(h)
            except Exception:
                pass

    # ------------------------------------------------------------------------------------------ helpers
    def rope(self, maxpos: int):
        if maxpos not in self._rope:
            self._rope[maxpos] = ops.rope_tables(maxpos, self.device)
        return self._rope[maxpos]

    def cached(self, key: tuple, make) -> torch.Tensor:
        # never evicted: captured CUDA graphs hold raw pointers to these tensors (a few KB per input signature)
        t = self._idx_cache.get(key)
        if t is None:
            t = make().to(self.device)
            self._idx_cache[key] = t
        return t

    def table(self, C_: int, h: int, w: int, aspect: float) -> torch.Tensor:
        key = (C_, h, w, round(aspect, 9))
        if key not in self._tables:
            self._tables[key] = uv_posembed_table(C_, h, w, aspect, self.device)
        return self._tables[key]

    def table_xy(self, C_: int, h: int, w: int, aspect: float):
        key = ("xy", C_, h, w, round(aspect, 9))
        if key not in self._tables:
            self._tables[key] = uv_posembed_separable(C_, h, w, aspect, self.device)
        return self._tables[key]

    def warm_tables(self, H: int, W: int):
        """Build the UV position-embedding tables of this image size on the CURRENT stream (the two DPT heads run on
        different streams and share the cached tables; the first use must not race with the copy that fills them)."""
        hp, wp = H // self.patch, W // self.patch
        for pk in self.dpt_packs.values():
            for oc in pk.oc:
                self.table(oc, hp, wp, W / H)
            self.table_xy(pk.feat // 2, hp * self.patch, wp * self.patch, W / H)

    def _workspace(self, name: str, nbytes: int) -> torch.Tensor:
        if nbytes < 0:
            raise L.OvgError("libovg: workspace size query failed")
        return self.ws.get(name, (nbytes,), torch.uint8)

    # ------------------------------------------------------------------------------------------ DINOv2 patchifier
    def dino_patchify(self, images: torch.Tensor, pos_embed: torch.Tensor, mean, std) -> torch.Tensor:
        """images fp32 [K,3,H,W] in [0,1] -> x_norm_patchtokens fp32 [K,P,C] (reference
        layers/vision_transformer.py:214-271).  pos_embed: fp32 [1, 1+P, C], already interpolated to this grid."""
        lib, d = L.lib(), self.dino
        K, _, H, W = images.shape
        P = (H // self.patch) * (W // self.patch)
        pe = self.m.aggregator.patch_embed
        # [cls + pos0, registers, pos_patches]: the same for every frame; the patch-embedding GEMM adds on top
        base = torch.cat([pe.cls_token.float() + pos_embed[:, :1], pe.register_tokens.float(), pos_embed[:, 1:]], 1).contiguous()
        wsb = self._workspace("dino_ws", lib.ovg_dino_workspace_bytes(self.h_dino, K, H, W))
        out = self.ws.get("dino_out", (K, P, self.C), F32)
        m3 = (C.c_float * 3)(*[float(v) for v in mean])
        s3 = (C.c_float * 3)(*[float(v) for v in std])
        img = images.contiguous()
        L.check(lib.ovg_dino_forward(self.h_dino, img.data_ptr(), base.data_ptr(), C.cast(m3, C.c_void_p), C.cast(s3, C.c_void_p),
                                     K, H, W, wsb.data_ptr(), wsb.numel(), out.data_ptr(), L.stream()))
        return out

    # ------------------------------------------------------------------------------------------ aggregator
    def aggregate(self, patch_tokens: torch.Tensor, inj: torch.Tensor, depth: Optional[torch.Tensor],
                  mask: Optional[torch.Tensor], depth_idx: List[int], B: int, S: int, H: int, W: int,
                  keep: Sequence[int], cp=None, views_total: int = 0):
        """patch_tokens fp32 [K,P,C]; inj fp32 [depth+1,K,C].  Returns ({layer: bf16 slot [K,T,2C]}, cam fp32 [K,2C]).
        ``cp`` (a ContextParallel): B = 1, S = this rank's views of a scene with ``views_total`` views."""
        lib = L.lib()
        Cc, R = self.C, self.R
        K = B * S
        hp, wp = H // self.patch, W // self.patch
        T = hp * wp + R + 1
        if max(hp, wp) > L.MAX_PATCHES_PER_SIDE:
            raise ValueError(f"{H}x{W} input: at most {L.MAX_PATCHES_PER_SIDE} patches per side are supported "
                             f"({L.MAX_PATCHES_PER_SIDE * self.patch} px at patch size {self.patch})")
        assert tuple(keep) == self.keep or set(keep) == set(self.keep), "kept layers are fixed when the engine is built"
        cos, sin = self.rope(max(hp, wp) + 1)
        Sd = len(depth_idx)
        idx = idx_loc = d32 = m32 = None
        n_loc = 0
        if Sd:
            # context parallel: depth / mask are the full [1, views_total, H, W] tensors, depth_idx the scene indices of all
            # selected views (the normalisation mean is global), and the rank embeds only the selected views it owns
            S_src = views_total if cp is not None else S
            idx = self.cached(("depth_idx", tuple(depth_idx)), lambda: torch.tensor(depth_idx, dtype=torch.int32))
            d32 = depth.reshape(B, S_src, H, W).to(F32).contiguous()
            m32 = mask.reshape(B, S_src, H, W).to(F32).contiguous()
            if cp is not None:
                v0, n = cp.local_views(views_total)
                loc = [i for i in depth_idx if v0 <= i < v0 + n]
                n_loc = len(loc)
                if n_loc:
                    idx_loc = self.cached(("depth_idx", tuple(loc)), lambda: torch.tensor(loc, dtype=torch.int32))
        wsb = self._workspace("agg_ws", lib.ovg_aggregator_workspace_bytes(self.h_agg, B, S, H, W, Sd))
        slot_t = [self.ws.get(f"slot{i}", (K, T, 2 * Cc)) for i in self.keep]
        slot_p = (C.c_void_p * 4)(*[t.data_ptr() for t in slot_t])
        cam_out = self.ws.get("cam_out", (K, 2 * Cc), F32)
        pt, ij = patch_tokens.contiguous(), inj.contiguous()
        if cp is not None:
            assert B == 1, "context parallelism shards the views of one scene"
            cd = cp.desc(self.heads, views_total * T, views_total)
            L.check(lib.ovg_aggregator_forward_cp(self.h_agg, C.byref(cd), pt.data_ptr(), ij.data_ptr(), L.ptr(d32), L.ptr(m32),
                                                  L.ptr(idx), Sd, L.ptr(idx_loc), n_loc, cos.data_ptr(), sin.data_ptr(),
                                                  cos.shape[0], S, H, W, wsb.data_ptr(), wsb.numel(), slot_p, cam_out.data_ptr(),
                                                  L.stream()))
        else:
            L.check(lib.ovg_aggregator_forward(self.h_agg, pt.data_ptr(), ij.data_ptr(), L.ptr(d32), L.ptr(m32), L.ptr(idx), Sd,
                                               cos.data_ptr(), sin.data_ptr(), cos.shape[0], B, S, H, W, wsb.data_ptr(),
                                               wsb.numel(), slot_p, cam_out.data_ptr(), L.stream()))
        return dict(zip(self.keep, slot_t)), cam_out

    # ------------------------------------------------------------------------------------------ camera head
    def camera_head(self, cam_tokens: torch.Tensor, B: int, S: int, iters: int = 4) -> List[torch.Tensor]:
        """cam_tokens fp32 [B*S, 2C] -> list of `iters` activated pose encodings fp32 [B, S, 9] (heads/camera_head.py:83-154)."""
        lib = L.lib()
        K = B * S
        wsb = self._workspace("cam.ws", lib.ovg_camera_workspace_bytes(self.h_cam, K))
        out = torch.empty(iters, K, 9, device=self.device, dtype=F32)
        ct = cam_tokens.contiguous()
        L.check(lib.ovg_camera_forward(self.h_cam, ct.data_ptr(), B, S, iters, out.data_ptr(), wsb.data_ptr(), wsb.numel(), L.stream()))
        return [out[i].view(B, S, 9) for i in range(iters)]

    # ------------------------------------------------------------------------------------------ DPT head
    def dpt_alloc(self, name: str, K: int, H: int, W: int):
        pk = self.dpt_packs[name]
        return (torch.empty(K, H, W, pk.outc - 1, device=self.device, dtype=F32),
                torch.empty(K, H, W, device=self.device, dtype=F32))

    def dpt(self, name: str, slots: Dict[int, torch.Tensor], layers: Sequence[int], K: int, H: int, W: int,
            head_act: int, chunk: int = 8, out=None):
        """One DPT head over all K frames in chunks of 8 (reference heads/dpt_head.py:153-183: results are chunk independent).
        Every head has its own workspace, so the two heads may run concurrently on different streams."""
        lib, pk = L.lib(), self.dpt_packs[name]
        preds, conf = out if out is not None else self.dpt_alloc(name, K, H, W)
        hp, wp = H // self.patch, W // self.patch
        T = hp * wp + self.R + 1
        slot_p = (C.c_void_p * 4)(*[slots[i].data_ptr() for i in layers])
        tabs = [self.table(oc, hp, wp, W / H) for oc in pk.oc]
        tab_p = (C.c_void_p * 4)(*[t.data_ptr() for t in tabs])
        tx, ty = self.table_xy(pk.feat // 2, hp * self.patch, wp * self.patch, W / H)
        fc_max = min(chunk, K)
        wsb = self._workspace(name + ".ws", lib.ovg_dpt_workspace_bytes(self.h_dpt[name], fc_max, H, W))
        for f0 in range(0, K, chunk):
            L.check(lib.ovg_dpt_forward(self.h_dpt[name], slot_p, T, self.R + 1, f0, min(chunk, K - f0), H, W, tab_p,
                                        tx.data_ptr(), ty.data_ptr(), head_act, preds.data_ptr(), conf.data_ptr(),
                                        wsb.data_ptr(), wsb.numel(), L.stream()))
        return preds, conf

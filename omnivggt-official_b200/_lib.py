"""ctypes binding of libovg.so (include/ovg.h).  There is NO fallback: if the shared library is missing or the
device is not a B200 the import / first call fails loudly."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("OVG_LIB_PATH") or os.path.join(_HERE, "libovg.so")   # override: A/B kernel builds

EPI_BF16, EPI_RESID, EPI_QKV, EPI_HEADTAIL = 0, 1, 2, 3
ROWS_IDENT, ROWS_DENSE2PAD, ROWS_PAD, ROWS_PIXSHUF = 0, 1, 2, 3
ACT_NONE, ACT_GELU, ACT_RELU = 0, 1, 2

_vp, _i, _ll, _f = C.c_void_p, C.c_int, C.c_longlong, C.c_float


class GemmArgs(C.Structure):
    """Mirror of ``ovg_gemm_args`` (include/ovg.h); field order must match exactly."""
    _fields_ = [
        ("a", _vp), ("a_rows", _ll), ("a_cols", _i), ("lda", _ll),
        ("b", _vp), ("n", _i), ("ldb", _ll),
        ("m", _i),
        ("num_taps", _i), ("tap_off", _i * 9),
        ("epi", _i),
        ("bias", _vp), ("act", _i), ("out", _vp), ("ldo", _ll),
        ("table", _vp), ("table_rows", _i),
        ("skip1", _vp), ("skip2", _vp),
        ("rowmap", _i), ("gh", _i), ("gw", _i), ("ps", _i), ("cout", _i),
        ("gamma", _vp), ("row_index", _vp),
        ("q_out", _vp), ("k_out", _vp), ("v_out", _vp),
        ("C", _i), ("ntok", _i), ("T", _i), ("nspecial", _i), ("wp", _i), ("maxpos", _i),
        ("qn_w", _vp), ("qn_b", _vp), ("kn_w", _vp), ("kn_b", _vp),
        ("rope_cos", _vp), ("rope_sin", _vp), ("qscale", _f),
        ("w2", _vp), ("b2", _vp), ("outc", _i), ("head_act", _i), ("preds", _vp), ("conf", _vp),
        ("block_n", _i), ("qk_norm", _i), ("rope", _i),
        ("k_peers", _vp * 8), ("v_peers", _vp * 8), ("n_peers", _i), ("peer_ntok", _i), ("peer_tok_off", _ll),
        ("f16", _i),
    ]


class BlockWeights(C.Structure):
    """Mirror of ``ovg_block_weights``."""
    _fields_ = [(n, _vp) for n in ("ln1_w", "ln1_b", "w_qkv", "b_qkv", "qn_w", "qn_b", "kn_w", "kn_b", "w_proj", "b_proj", "g1",
                                   "ln2_w", "ln2_b", "w_fc1", "b_fc1", "w_fc2", "b_fc2", "g2")]


class AggregatorDesc(C.Structure):
    """Mirror of ``ovg_aggregator_desc``."""
    _fields_ = [("C", _i), ("registers", _i), ("depth", _i), ("patch", _i),
                ("frame_blocks", C.POINTER(BlockWeights)), ("global_blocks", C.POINTER(BlockWeights)),
                ("cam_tok", _vp), ("reg_tok", _vp), ("placeholder", _vp), ("depth_w", _vp), ("depth_b", _vp), ("ones_c", _vp),
                ("keep_layers", _i * 4)]


class DinoDesc(C.Structure):
    """Mirror of ``ovg_dino_desc``."""
    _fields_ = [("C", _i), ("registers", _i), ("depth", _i), ("patch", _i), ("kpad", _i),
                ("blocks", C.POINTER(BlockWeights)), ("w_patch", _vp), ("b_patch", _vp), ("norm_w", _vp), ("norm_b", _vp),
                ("ones_c", _vp)]


class DptFusion(C.Structure):
    """Mirror of ``ovg_dpt_fusion``."""
    _fields_ = [("rcu1", _vp * 4), ("rcu2", _vp * 4), ("oc_w", _vp), ("oc_b", _vp)]


class DptDesc(C.Structure):
    """Mirror of ``ovg_dpt_desc``."""
    _fields_ = [("C2", _i), ("feat", _i), ("patch", _i), ("outc", _i), ("oc", _i * 4),
                ("proj_w", _vp * 4), ("proj_b", _vp * 4), ("up_w", _vp * 2), ("up_b", _vp * 2), ("down_w", _vp), ("down_b", _vp),
                ("rn_w", _vp * 4), ("fus", DptFusion * 4), ("oc1_w", _vp), ("oc1_b", _vp), ("oc2_w", _vp), ("oc2_b", _vp),
                ("w2", _vp), ("b2", _vp), ("f16", _i)]


class CameraDesc(C.Structure):
    """Mirror of ``ovg_camera_desc``."""
    _fields_ = [("D", _i), ("heads", _i), ("trunk_depth", _i), ("trunk", C.POINTER(BlockWeights)),
                ("token_norm_w", _vp), ("token_norm_b", _vp), ("trunk_norm_w", _vp), ("trunk_norm_b", _vp), ("empty_pose", _vp),
                ("embed_w", _vp), ("embed_b", _vp), ("mod_w", _vp), ("mod_b", _vp), ("fc1_w", _vp), ("fc1_b", _vp),
                ("fc2_w", _vp), ("fc2_b", _vp)]


class ContextParallelDesc(C.Structure):
    """Mirror of ``ovg_context_parallel``."""
    _fields_ = [("rank", _i), ("world", _i), ("views_total", _i), ("k_peers", (_vp * 8) * 2), ("v_peers", (_vp * 8) * 2),
                ("flag_peers", _vp * 8), ("epoch_counter", _vp), ("cam_peers", _vp * 8)]


_pp = C.POINTER(_vp)
EXPORTS = {
    "ovg_version": (C.c_int, []),
    "ovg_last_error": (C.c_char_p, []),
    "ovg_device_check": (C.c_int, []),
    "ovg_launch_count": (C.c_longlong, []),
    "ovg_gemm": (C.c_int, [C.POINTER(GemmArgs), _vp]),
    "ovg_attention": (C.c_int, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "ovg_attention_kv": (C.c_int, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "ovg_attention_scratch_bytes": (C.c_longlong, []),
    "ovg_attention_kv_ws": (C.c_int, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _ll, _vp]),
    "ovg_peer_barrier": (C.c_int, [C.POINTER(_vp), _vp, _i, _i, _vp]),
    "ovg_aggregator_forward_cp": (C.c_int, [_vp, C.POINTER(ContextParallelDesc), _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _vp, _vp, _i,
                                            _i, _i, _i, _vp, _ll, _pp, _vp, _vp]),
    "ovg_depth_im2col2": (C.c_int, [_vp, _vp, _vp, _i, _vp, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "ovg_layernorm": (C.c_int, [_vp, _i, _ll, _vp, _i, _ll, _i, _i, _vp, _vp, _f, _i, _i, _i, _vp]),
    "ovg_image_im2col": (C.c_int, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "ovg_assemble_tokens": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "ovg_inject_snapshot": (C.c_int, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "ovg_depth_im2col": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "ovg_im2col3x3s2": (C.c_int, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "ovg_dpt_tail_supported": (C.c_int, [_i, _i, _i, _i, _i]),
    "ovg_dpt_tail_scratch_bytes": (C.c_longlong, [_i, _i]),
    "ovg_dpt_tail": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "ovg_upsample_bilinear": (C.c_int, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "ovg_preprocess_image": (C.c_int, [_vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "ovg_preprocess_depth": (C.c_int, [_vp, _ll, _ll, _vp, _vp, _i, _i, _i, _f, _vp, _vp, _vp]),
    "ovg_prepare_cameras": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "ovg_pose_decode": (C.c_int, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "ovg_unproject_depth": (C.c_int, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "ovg_conf_percentile_mask": (C.c_int, [_vp, _ll, _f, _f, _vp, _vp, _vp, _vp, _vp]),
    # ---- runtime (handle-level sequences)
    "ovg_aggregator_create": (C.c_int, [C.POINTER(AggregatorDesc), _pp]),
    "ovg_aggregator_destroy": (None, [_vp]),
    "ovg_aggregator_workspace_bytes": (_ll, [_vp, _i, _i, _i, _i, _i]),
    "ovg_aggregator_forward": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _i, _i, _i, _i, _i, _vp, _ll, _pp, _vp, _vp]),
    "ovg_dino_create": (C.c_int, [C.POINTER(DinoDesc), _pp]),
    "ovg_dino_destroy": (None, [_vp]),
    "ovg_dino_workspace_bytes": (_ll, [_vp, _i, _i, _i]),
    "ovg_dino_forward": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _ll, _vp, _vp]),
    "ovg_dpt_create": (C.c_int, [C.POINTER(DptDesc), _pp]),
    "ovg_dpt_destroy": (None, [_vp]),
    "ovg_dpt_workspace_bytes": (_ll, [_vp, _i, _i, _i]),
    "ovg_dpt_forward": (C.c_int, [_vp, _pp, _i, _i, _i, _i, _i, _i, _pp, _vp, _vp, _i, _vp, _vp, _vp, _ll, _vp]),
    "ovg_camera_create": (C.c_int, [C.POINTER(CameraDesc), _pp]),
    "ovg_camera_destroy": (None, [_vp]),
    "ovg_camera_workspace_bytes": (_ll, [_vp, _i]),
    "ovg_camera_forward": (C.c_int, [_vp, _vp, _i, _i, _i, _vp, _vp, _ll, _vp]),
    "ovg_runtime_time_attention": (None, [_i]),
    "ovg_runtime_attention_split": (None, [_i]),
    "ovg_runtime_attention_times": (C.c_int, [_vp, _i]),
}
PERCENTILE_WORKSPACE_BYTES = 6 * 8 + 512 * 4 + 4 * 4
MAX_PATCHES_PER_SIDE = 146            # OVG_MAX_PATCHES_PER_SIDE (include/ovg.h): 2 044 px per side at patch 14


def DEPTH_SCRATCH_DOUBLES(B: int) -> int:
    """Mirror of OVG_DEPTH_SCRATCH_DOUBLES (include/ovg.h)."""
    return B * (2 * 1024 + 1)

_lib: Optional[C.CDLL] = None
_device_ok = False


class OvgError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load libovg.so and bind every symbol declared in include/ovg.h (no GPU needed for this step)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise OvgError(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU / PyTorch fallback for the hot path)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in EXPORTS.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def lib() -> C.CDLL:
    """Library handle for compute calls: additionally requires a B200 as the current device."""
    global _device_ok
    l = load()
    if not _device_ok:
        if not torch.cuda.is_available():
            raise OvgError("libovg needs a CUDA device (B200); torch.cuda.is_available() is False")
        torch.cuda.current_device()          # make sure the primary context exists
        check(l.ovg_device_check())
        _device_ok = True
    return l


def check(rc: int) -> None:
    if rc != 0:
        raise OvgError(f"libovg error {rc}: {load().ovg_last_error().decode()}")


def ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream

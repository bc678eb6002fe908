"""Images above 882 px per side (CPU): the boundary module hands the runtime a RoPE table with more than 64 rows, sizes past
the supported envelope (146 patches per side, include/ovg.h) are refused with a message naming the limit, and the host
oracle of the loader matches the unmodified reference loader at ``target_size=1036``."""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import preprocess_oracle as PO
from oracle.synth import make_inputs
from oracle.synth_folder import FOLDERS, make_folder
from test_dryrun_cpu import dry  # noqa: F401  (fixture)
from test_host_cpu import mini_model
from test_preprocess import _read_folder

GOLD = json.load(open(os.path.join(GOLDEN, "preprocess_hires.json")))


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _record_args(rec, name):
    """Wrap the recorder so that the arguments of `name` are kept as well."""
    seen = []
    fn = rec.__getattr__(name)

    def wrapped(*a):
        seen.append(a)
        return fn(*a)
    setattr(rec, name, wrapped)
    return seen


def test_wide_forward_reaches_the_runtime_with_75_rope_rows(dry):
    from omnivggt_official_b200.engine import Engine
    m = mini_model().eval()
    m._engine = Engine(m)
    agg = _record_args(dry, "ovg_aggregator_forward")
    inp = make_inputs(1, 2, 784, 1036, seed=3)
    out = m(images=inp["images"])
    assert out["depth"].shape == (1, 2, 784, 1036, 1) and out["world_points"].shape == (1, 2, 784, 1036, 3)
    assert len(agg) == 1
    a = agg[0]
    maxpos, B, S, H, W = a[9:14]
    assert (maxpos, B, S, H, W) == (1036 // 14 + 1, 1, 2, 784, 1036) and maxpos == 75


def test_one_patch_past_the_envelope_is_refused(dry):
    from omnivggt_official_b200 import _lib
    from omnivggt_official_b200.engine import Engine
    m = mini_model().eval()
    m._engine = Engine(m)
    too_tall = 14 * (_lib.MAX_PATCHES_PER_SIDE + 1)
    with pytest.raises(ValueError, match=r"at most 146 patches per side .*2044 px"):
        m(images=make_inputs(1, 1, too_tall, 28, seed=3)["images"])
    assert dry.calls.count("ovg_aggregator_forward") == 0
    out = m(images=make_inputs(1, 1, 14 * _lib.MAX_PATCHES_PER_SIDE, 28, seed=3)["images"])   # the edge itself is accepted
    assert out["depth"].shape == (1, 1, 2044, 28, 1) and dry.calls.count("ovg_aggregator_forward") == 1


@pytest.mark.parametrize("name", sorted(FOLDERS))
def test_oracle_matches_reference_loader_at_1036(name, tmp_path):
    import PIL
    if PIL.__version__ != GOLD["_versions"]["pillow"]:
        pytest.skip("fixture hashes are for the pinned Pillow build")
    g = GOLD[name]
    imgs, cams, deps, tr = _read_folder(make_folder(str(tmp_path), name, seed=0))
    deps = [d.T if t else d for d, t in zip(deps, tr)]          # the reference transposes PNG depth (visual_util.py:771)
    images, extr, intr, dep, mask, didx, cidx = PO.load_views(imgs, cams, deps, target_size=GOLD["_target_size"])
    assert list(images.shape) == g["images_shape"] and didx == g["depth_indices"] and cidx == g["camera_indices"]
    assert max(images.shape[-2:]) == 1036 and images.shape[-1] == 1036
    assert _sha(images.astype(np.float32)) == g["images_f32_sha256"]
    assert _sha(dep.astype(np.float32)) == g["depth_sha256"] and _sha(mask.astype(np.float32)) == g["mask_sha256"]
    assert np.allclose(extr, np.array(g["extrinsics"]), atol=2e-6) and np.allclose(intr, np.array(g["intrinsics"]), rtol=1e-5, atol=1e-3)

"""tests/golden/preprocess_hires.json: the UNMODIFIED reference loader (visual_util.py:679-841 load_images_and_cameras) at
``target_size=1036`` on the seeded synthetic folders of oracle/synth_folder.py -- both folders are upscaled there: 640 x 480
becomes 784 x 1036, 300 x 500 is resized to 1036 x 1726 and cropped to 1036 x 1036 (build container only; TEST INFRASTRUCTURE).

    python oracle/make_golden_pre_hires.py
"""
from __future__ import annotations

import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle.make_golden_pre import GOLDEN, summarize  # noqa: E402
from oracle.ref_shims import REFERENCE_ROOT  # noqa: E402
from oracle.synth_folder import FOLDERS, make_folder  # noqa: E402

TARGET_SIZE = 1036


def main():
    import importlib.machinery
    from unittest.mock import MagicMock
    # the same import stubs as oracle/make_golden_pre.py (viewer / evaluation dependencies the loader never calls)
    for mod in ("evo", "evo.main_ape", "evo.main_rpe", "evo.core", "evo.core.sync", "evo.core.metrics", "evo.core.trajectory",
                "evo.tools", "evo.tools.file_interface", "evo.tools.plot", "matplotlib", "matplotlib.pyplot", "onnxruntime", "trimesh",
                "viser", "viser.transforms", "pillow_heif", "imageio", "imageio.v2", "imageio.v3"):
        m = MagicMock()
        m.__spec__ = importlib.machinery.ModuleSpec(mod, None)
        m.__name__, m.__path__ = mod, []
        sys.modules.setdefault(mod, m)
    sys.path.insert(0, REFERENCE_ROOT)
    import visual_util as vu
    res = {"_target_size": TARGET_SIZE}
    with tempfile.TemporaryDirectory() as root:
        for name in FOLDERS:
            d = make_folder(root, name, seed=0)
            out = vu.load_images_and_cameras(d["images"], d["cameras"], d["depths"], target_size=TARGET_SIZE)
            res[name] = summarize([t.numpy() if hasattr(t, "numpy") else t for t in out])
            print(name, res[name]["images_shape"], res[name]["depth_indices"], res[name]["camera_indices"])
    import PIL
    import cv2
    res["_versions"] = {"pillow": PIL.__version__, "opencv": cv2.__version__}
    with open(os.path.join(GOLDEN, "preprocess_hires.json"), "w") as f:
        json.dump(res, f, indent=0, sort_keys=True)


if __name__ == "__main__":
    main()

"""bench.py contract checks that need no GPU: the reference (CPU) arm prints one JSON line with the agreed keys on rank 0
only, and drops torchrun's OMP_NUM_THREADS=1 before torch initialises its thread pools."""
import argparse
import importlib.util
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("ovg_bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_reference_arm_line(monkeypatch, capsys):
    from oracle import cpu_baseline as cb
    from oracle import vendor_ref
    monkeypatch.setattr(cb, "sample", lambda *a, **k: (70.0, {}))       # one sample costs ~1 min on 8 cores: stubbed
    monkeypatch.setattr(vendor_ref, "OUT", "/nonexistent/ref.zip")     # exercise the labelled fallback (no 1-minute forwards)
    bench = _bench()
    args = argparse.Namespace(gpus=2, steps=3, warmup=1, impl="reference", config="cfg2", no_cpu_baseline=False)
    bench.run_reference(args, 1, 2)                                      # non-zero ranks: no work, no output
    assert capsys.readouterr().out.strip() == ""
    bench.run_reference(args, 0, 2)
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "view_sets_per_sec" and line["unit"] == "view-sets/s"
    assert line["n_gpus"] == 2 and line["steps"] == 3 and line["higher_is_better"] is True and line["gpu_launches"] == 0
    assert abs(line["value"] - 1 / 70.0) < 1e-9 and abs(line["ms_per_step"] - 70e3) < 1e-6
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "view-sets/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and line["config"]["name"] == "cfg2"
    assert line["cpu_baseline"]["sample"].startswith("FALLBACK")


def test_reference_arm_runs_the_packed_reference(monkeypatch, capsys):
    """With oracle/_ref present the arm times whole forwards of the unmodified reference class (stubbed here by a tiny
    module with the same call signature: the real one needs a minute per forward) and reports the forwards actually run."""
    import torch
    from oracle import vendor_ref

    class Tiny(torch.nn.Module):
        calls = 0

        def forward(self, images, extrinsics, intrinsics, depth, mask, depth_gt_index, camera_gt_index):
            Tiny.calls += 1
            assert images.shape == (1, 4, 3, 518, 518) and depth_gt_index == [] and camera_gt_index == []
            return {}

    monkeypatch.setattr(vendor_ref, "import_reference_zip", lambda: Tiny)
    bench = _bench()
    args = argparse.Namespace(gpus=1, steps=3, warmup=1, impl="reference", config="cfg1", no_cpu_baseline=False)
    bench.run_reference(args, 0, 1)
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert Tiny.calls == 4 and line["steps"] == 3 and line["warmup"] == 1
    assert line["cpu_baseline"]["kind"] == "reference" and "unmodified reference" in line["cpu_baseline"]["sample"]
    assert line["config"]["name"] == "cfg1" and line["e2e"]["value"] == line["value"]


def test_configs_follow_baseline_json():
    bench = _bench()
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert len(base["configs"]) == 5 and sorted(bench.CONFIGS) == ["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"]
    assert bench.CONFIGS["cfg1"]["S"] == 4 and bench.CONFIGS["cfg2"]["S"] == 8 and bench.CONFIGS["cfg5"]["S"] == 24
    assert bench.CONFIGS["cfg3"]["depth_idx"] == list(range(8)) == bench.CONFIGS["cfg3"]["cam_idx"]
    assert bench.CONFIGS["cfg4"]["scenes"] == 32 and bench.CONFIGS["cfg4"]["scaling"] == "strong"
    c5 = bench.CONFIGS["cfg5"]
    assert 0 in c5["cam_idx"] and 0 < len(c5["depth_idx"]) < 24 and 0 < len(c5["cam_idx"]) < 24     # partial; view 0 has a camera
    inp = bench.synth_inputs(1, 2, seed=3)
    assert inp["images"].shape == (1, 2, 3, 518, 518) and inp["depth"].shape == (1, 2, 518, 518, 1)
    import torch
    R = inp["extrinsics"][0, :, :, :3]
    assert torch.allclose(R @ R.transpose(-1, -2), torch.eye(3).expand(2, 3, 3), atol=1e-5) and (torch.linalg.det(R) > 0).all()


def test_dump_outputs_whole_and_sampled(tmp_path):
    """--dump-outputs: one float32 .npy per returned array with the forward calls of the step concatenated, the input echo and
    non-tensors left out; over the size cap the small arrays stay whole and the large ones become the same sample every run."""
    import numpy as np
    import torch
    bench = _bench()
    g = torch.Generator().manual_seed(0)

    def call():
        return {"pose_enc": torch.randn(2, 3, 9, generator=g), "pose_enc_list": [torch.randn(2, 3, 9, generator=g) for _ in range(2)],
                "depth": torch.rand(2, 3, 40, 50, 1, generator=g), "world_points": torch.randn(2, 3, 40, 50, 3, generator=g).double(),
                "images": torch.rand(2, 3, 3, 40, 50, generator=g), "view_range": (0, 3)}

    outs = [call(), call()]
    whole = {"pose_enc": torch.cat([o["pose_enc"] for o in outs]), "depth": torch.cat([o["depth"] for o in outs]),
             "world_points": torch.cat([o["world_points"] for o in outs]).float(),
             **{f"pose_enc_list.{i}": torch.cat([o["pose_enc_list"][i] for o in outs]) for i in range(2)}}
    bench.dump_outputs(outs, str(tmp_path / "all"))
    assert sorted(p.name for p in (tmp_path / "all").iterdir()) == sorted(k + ".npy" for k in whole)
    for k, v in whole.items():
        a = np.load(tmp_path / "all" / f"{k}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, v.numpy()), k

    limit = 100_000                                     # depth 96 000 B + world_points 288 000 B + 3 x 432 B
    for d in ("s1", "s2"):
        bench.dump_outputs(outs, str(tmp_path / d), limit=limit)
    got = {k: np.load(tmp_path / "s1" / f"{k}.npy") for k in whole}
    assert sum(a.nbytes for a in got.values()) <= limit
    for k in ("pose_enc", "pose_enc_list.0", "pose_enc_list.1"):
        assert np.array_equal(got[k], whole[k].numpy()), k
    for k in ("depth", "world_points"):
        assert got[k].ndim == 1 and 0.4 * limit / 4 < got[k].size < whole[k].numel(), (k, got[k].size)
        assert got[k].dtype == np.float32 and np.isin(got[k], whole[k].numpy()).all()
        assert np.array_equal(got[k], np.load(tmp_path / "s2" / f"{k}.npy")), k


def test_reference_arm_ignores_torchrun_thread_cap():
    """torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU arm must still see every core."""
    # run the arm in a fresh interpreter with the caps exported and the (slow) sample stubbed
    driver = ("import os, sys, json, argparse, importlib.util\n"
              f"sys.path.insert(0, {ROOT!r})\n"
              f"spec = importlib.util.spec_from_file_location('b', {os.path.join(ROOT, 'bench.py')!r})\n"
              "b = importlib.util.module_from_spec(spec); spec.loader.exec_module(b)\n"
              "assert 'torch' not in sys.modules, 'bench.py must not import torch before the reference arm cleans the environment'\n"
              "import types\n"
              "stub = types.ModuleType('oracle.cpu_baseline'); stub.sample = lambda *a, **k: (70.0, {}); stub.SAMPLE_DESC = 'stub'\n"
              "import oracle; sys.modules['oracle.cpu_baseline'] = stub; oracle.cpu_baseline = stub\n"
              "import oracle.vendor_ref as vr; vr.OUT = '/nonexistent/ref.zip'\n"
              "b.run_reference(argparse.Namespace(gpus=1, steps=1, warmup=0, impl='reference', config='cfg2', no_cpu_baseline=False), 0, 1)\n")
    env = dict(os.environ, OMP_NUM_THREADS="1", MKL_NUM_THREADS="1")
    out = subprocess.run([sys.executable, "-c", driver], env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    if ncpu > 1:
        assert line["cpu_baseline"]["cores"] > 1, line["cpu_baseline"]

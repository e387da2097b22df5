"""bench.py --dump-outputs: the arrays the timed step returned in its last step, as float32 .npy files within 64 MB."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_samples_the_same_rows_within_the_budget(tmp_path):
    import bench
    g = torch.Generator().manual_seed(0)
    arrays = {"rgb": torch.randn(8, 4096, 32, generator=g), "depth": torch.randn(8, 4096, 1, generator=g, dtype=torch.float64),
              "loss": torch.tensor(3.5), "bias": torch.randn(64, generator=g), "grad": torch.randn(400000, generator=g)}
    budget = 2 << 20
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays, budget=budget)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["bias.npy", "depth.npy", "grad.npy", "loss.npy", "rgb.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= budget
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float32 and np.array_equal(a, b), f
    # arrays of up to 1 MB are stored whole
    assert np.array_equal(np.load(tmp_path / "a" / "depth.npy"), arrays["depth"].float().numpy())
    assert np.load(tmp_path / "a" / "loss.npy") == np.float32(3.5)
    # the 4 MB map keeps whole rows of the original, in order
    orig = arrays["rgb"].reshape(-1, 32).numpy()
    kept = np.load(tmp_path / "a" / "rgb.npy")
    assert kept.shape[1] == 32 and orig.shape[0] // 4 < kept.shape[0] < orig.shape[0]
    row_of = {r.tobytes(): i for i, r in enumerate(orig)}
    idx = np.array([row_of[r.tobytes()] for r in kept])
    assert np.all(np.diff(idx) > 0) and np.array_equal(orig[idx], kept)
    # a vector over 1 MB keeps elements, the same fraction as the map's rows
    grad = np.load(tmp_path / "a" / "grad.npy")
    assert grad.shape[1] == 1 and abs(grad.shape[0] / 400000 - kept.shape[0] / orig.shape[0]) < 1e-3
    # rows wider than an array's share: elements are sampled instead, still within the budget
    bench.dump_outputs(str(tmp_path / "w"), {"wide": torch.randn(2, 600000, generator=g), "rgb": arrays["rgb"]}, budget=budget)
    assert np.load(tmp_path / "w" / "wide.npy").shape[1] == 1
    assert sum(os.path.getsize(tmp_path / "w" / f) for f in os.listdir(tmp_path / "w")) <= budget
    with pytest.raises(ValueError, match="budget"):
        bench.dump_outputs(str(tmp_path / "d"), arrays, budget=100000)
    # within the default budget nothing is sampled
    bench.dump_outputs(str(tmp_path / "c"), arrays)
    assert np.array_equal(np.load(tmp_path / "c" / "rgb.npy"), arrays["rgb"].numpy())


@pytest.mark.gpu
def test_bench_dumps_what_the_timed_step_rendered(tmp_path):
    """The dump of a short c1 run is the render of bench.make_inputs' seeded inputs, and --steps sets the timed steps: the
    library launches of a 3-step run are three times those of a 1-step run."""
    import bench
    from nerffaceediting_b200.ray_sampler import RaySampler
    from nerffaceediting_b200.renderer import DisentangledImportanceRenderer
    from nerffaceediting_b200.triplane import denormalize_plane, normalize_plane
    out = tmp_path / "dump"

    def run(steps, *extra):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c1", "--steps", str(steps), "--warmup", "3",
                            "--no-extras", "--no-cpu-baseline", *extra], capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-2000:]
        return json.loads(r.stdout.strip().splitlines()[-1])
    one, three = run(1), run(3, "--dump-outputs", str(out))
    assert one["steps"] == 1 and three["steps"] == 3
    assert one["gpu_launches"] > 0 and three["gpu_launches"] == 3 * one["gpu_launches"]
    wl = bench.WORKLOADS["c1"]
    dev = torch.device("cuda:0")
    raw_host, dec, c2w, k, opts = bench.make_inputs(torch, wl, torch.device("cpu"), 1000)
    opts.update(nfe_precision="bf16x3", nfe_single_gather=True)
    mods = {"sampler": RaySampler(), "normalize_plane": normalize_plane, "denormalize_plane": denormalize_plane,
            "renderer": DisentangledImportanceRenderer(), "swap": False}
    with torch.no_grad():
        want = bench.hot_path_step(torch, mods, raw_host.to(dev), dec.to(dev), c2w.to(dev), k.to(dev), wl["res"], opts)
    assert sorted(os.listdir(out)) == ["depth.npy", "rgb.npy", "seg.npy", "wsum.npy"]
    for name, w in zip(("rgb", "seg", "depth", "wsum"), want):
        got = np.load(out / f"{name}.npy")
        w = w.cpu().numpy()
        assert got.dtype == np.float32 and got.shape == w.shape, name
        np.testing.assert_allclose(got, w, rtol=1e-5, atol=1e-6 * float(np.abs(w).max()), err_msg=name)

"""bench.py --dump-outputs: the arrays the timed path returned in its last step, in a form two builds can be compared by."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import REPO, native_scene, params_for


def test_dump_outputs_keeps_a_fixed_sample_of_a_large_image(tmp_path):
    import bench
    rng = np.random.default_rng(1)
    h, w = 1000, 1100                                        # more pixels than DUMP_PIXELS, like the 4K default workload
    rgb = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    sums = rng.random((h, w, 3), dtype=np.float32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), rgb, sums)
    names = ("image", "sum", "pixel_index")
    got = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in names}
    idx = got["pixel_index"].astype(np.int64)
    assert got["pixel_index"].dtype == np.float64 and np.array_equal(idx, got["pixel_index"])
    assert len(idx) == bench.DUMP_PIXELS and np.all(np.diff(idx) > 0) and 0 <= idx[0] and idx[-1] < h * w
    assert got["image"].dtype == np.float32 and np.array_equal(got["image"], rgb.reshape(-1, 3)[idx])
    assert got["sum"].dtype == np.float32 and np.array_equal(got["sum"], sums.reshape(-1, 3)[idx])
    assert sum(os.path.getsize(tmp_path / "a" / f"{n}.npy") for n in names) <= 64_000_000
    for n in names:                                          # the same pixels on every run
        assert np.array_equal(np.load(tmp_path / "b" / f"{n}.npy"), got[n])


@pytest.mark.gpu
def test_bench_dumps_what_its_last_timed_step_rendered(tmp_path):
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--workload", "cornell_box", "--width", "64", "--height", "48",
                        "--spp", "8", "--steps", "2", "--warmup", "1", "--no-per-config", "--no-cpu-baseline", "--dump-outputs", str(out)],
                       capture_output=True, text=True, cwd=tmp_path, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["config"]["width"] == 64 and line["config"]["spp_total"] == 8
    assert sorted(os.listdir(out)) == ["image.npy", "sum.npy"]
    image, sums = np.load(out / "image.npy"), np.load(out / "sum.npy")
    assert image.dtype == sums.dtype == np.float32 and image.shape == sums.shape == (48, 64, 3)
    ns = native_scene("cornell_box")
    rgb, s, _ = ns.render(params_for("cornell_box", 64, 48, 8, seed=1))
    ns.close()
    assert np.array_equal(image, rgb.astype(np.float32))
    assert np.allclose(sums, s, rtol=1e-5, atol=1e-6)

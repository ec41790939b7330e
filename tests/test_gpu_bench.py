"""bench.py --dump-outputs on the GPU: one file per output, float32 / float64, seeded samples of large arrays, and the
same outputs from two runs whatever the number of untimed settle steps -- `-m gpu`."""
import io
import json
import os
import sys
from contextlib import redirect_stdout

import numpy as np
import pytest

import bench

pytestmark = pytest.mark.gpu


def _run(monkeypatch, out, settle):
    monkeypatch.setattr(sys, "argv", ["bench.py", "--workload", "colonoscopy256", "--frames", "40", "--resolution", "64", "--steps", "3",
                                      "--warmup", "1", "--settle", str(settle), "--no-cpu-baseline", "--no-extras", "--dump-outputs", str(out)])
    monkeypatch.delenv("RANK", raising=False)
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    buf = io.StringIO()
    with redirect_stdout(buf):
        bench.main()
    lines = [l for l in buf.getvalue().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0]), {f[:-4]: np.load(os.path.join(out, f)) for f in sorted(os.listdir(out))}


def test_dump_outputs_are_reproducible(cuda, monkeypatch, tmp_path):
    monkeypatch.setattr(bench, "DUMP_VOXELS", 5000)          # 64^3 voxels: exercise the seeded sample
    line, a = _run(monkeypatch, tmp_path / "a", 0.0)
    _, b = _run(monkeypatch, tmp_path / "b", 0.5)
    assert line["steps"] == 3
    assert set(a) == {"tsdf", "weight", "update_counts", "mesh_vertices", "mesh_triangles"}
    assert a["tsdf"].shape == a["weight"].shape == (5000,)
    assert a["update_counts"].shape == (40,) and a["update_counts"].min() > 0
    assert a["mesh_vertices"].shape == (line["details"]["mc_vertices"], 3) and line["details"]["mc_triangles"] > 0
    assert a["mesh_triangles"].shape == (line["details"]["mc_triangles"], 3)
    assert all(x.dtype in (np.float32, np.float64) for x in a.values())
    assert sum(x.nbytes for x in a.values()) <= 64e6
    # 1 warm-up + 3 timed steps of 40 frames, each voxel updated at most once per frame
    assert a["weight"].max() > 0 and a["weight"].max() <= 4 * 40
    for k in a:
        assert np.array_equal(a[k], b[k]), k

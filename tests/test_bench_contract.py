"""bench.py contract checks that need no GPU: the reference arm's JSON line (keys, units, identical `config` dict in both
arms) and the workload table."""
import io
import json
import os
import sys
from contextlib import redirect_stdout

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    sys.path.insert(0, ROOT)
    import bench
    return bench


def test_reference_arm_prints_one_contract_line(monkeypatch):
    bench = _bench()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-budget", "0.5",
                                      "--workload", "colonoscopy256"])
    monkeypatch.delenv("RANK", raising=False)
    buf = io.StringIO()
    with redirect_stdout(buf):
        bench.main()
    lines = [l for l in buf.getvalue().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["scalable_fps"] > 0 and cb["scalable_open3d_schedule_fps"] > 0
    assert "colonoscopy256" in d["config"]["workload"] and d["config"]["resolution"] == 256 and d["vs_baseline"] is None
    # the GPU arm builds its `config` from the same function and arguments: identical dicts
    args = bench.parse()
    cfg, F, E, res, vl, trunc = bench.workload(args)
    assert bench.config_dict(args, F, cfg["W"], cfg["H"], res, vl, trunc) == d["config"]


def test_reference_arm_is_silent_on_other_ranks(monkeypatch):
    bench = _bench()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--gpus", "8", "--steps", "1", "--warmup", "1"])
    monkeypatch.setenv("RANK", "3")
    buf = io.StringIO()
    with redirect_stdout(buf):
        bench.main()
    assert buf.getvalue() == ""


def test_steps_and_dump_outputs_arguments_are_checked(monkeypatch):
    bench = _bench()
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"], ["--emulate-shard", "0/2", "--dump-outputs", "out"]):
        monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
        with pytest.raises(SystemExit):
            bench.parse()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "7", "--dump-outputs", "out"])
    args = bench.parse()
    assert args.steps == 7 and args.dump_outputs == "out"


def test_workload_table_covers_the_baseline_configs():
    bench = _bench()
    assert set(bench.WORKLOADS) == {"laparoscopy512", "colonoscopy256", "gastroscopy1024"}
    assert bench.metric_name(512) == "fused frames/s (640x480 depth -> 512^3 TSDF)"
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert "512" in base["metric"] and len(base["configs"]) == 5

"""bench.py contract checks that need no GPU: the reference arm's JSON line (oracle port on the host cores) and the
shape of the shared workload config."""
import io
import json
import os
import sys
import types
from contextlib import redirect_stdout

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    sys.path.insert(0, ROOT)
    import importlib
    return importlib.import_module("bench")


def test_reference_arm_line(monkeypatch):
    bench = _bench()
    monkeypatch.setattr(bench, "B_PRED", 48)  # a bounded sample of the same workload, small enough for the CPU suite
    args = types.SimpleNamespace(gpus=1, steps=2, warmup=1)
    buf = io.StringIO()
    with redirect_stdout(buf):
        bench.run_reference(args, rank=0, world=1)
    lines = [l for l in buf.getvalue().splitlines() if l.strip()]
    assert len(lines) == 1  # ONE JSON line
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["unit"] == bench.UNIT
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config"):
        assert k in d, k
    assert d["value"] > 0 and d["steps"] == 2 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["config"]["workload"].startswith("ncmapss_lrt Inception BNN predict")
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # the other ranks of a torchrun launch print nothing
    buf = io.StringIO()
    with redirect_stdout(buf):
        bench.run_reference(args, rank=1, world=2)
    assert buf.getvalue() == ""


def test_dump_outputs_files(tmp_path):
    bench = _bench()
    m = (torch.arange(4.0), torch.ones(4), torch.zeros(4), torch.full((4,), 2.0))
    bench.dump_outputs(str(tmp_path / "one"), dict(zip(("pred", "std", "ep_var", "al_var"), m)), rank=0, world=1)
    assert sorted(os.listdir(tmp_path / "one")) == ["al_var.npy", "ep_var.npy", "pred.npy", "std.npy"]
    got = np.load(tmp_path / "one" / "pred.npy")
    assert got.dtype == np.float32 and got.tolist() == [0.0, 1.0, 2.0, 3.0]
    bench.dump_outputs(str(tmp_path / "two"), {"pred": m[0]}, rank=1, world=2)
    assert os.listdir(tmp_path / "two") == ["pred_rank1.npy"]


def test_bad_arguments_stop_before_any_gpu_work(monkeypatch, capsys):
    bench = _bench()
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
        with pytest.raises(SystemExit) as e:
            bench.main()
        assert e.value.code == 2
    assert capsys.readouterr().out == ""


def test_both_arms_share_the_workload_config():
    bench = _bench()
    a, b = bench.workload_config("tc", 1), bench.workload_config("cpu", 8)
    assert a["workload"] == b["workload"] and "configs[0]" in a["workload"]
    assert a["windows_per_step_per_gpu"] == bench.B_PRED and a["mc_samples"] == bench.S_PRED
    assert "model" not in a  # names the workload, no model keys

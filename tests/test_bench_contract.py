"""bench.py contract pieces that can be checked without a GPU."""
import importlib.util
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load_bench():
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_reference_arm_reports_unavailable_without_cuda():
    import torch

    if torch.cuda.is_available():
        return  # on a GPU box the arm really runs; the driver exercises it
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference"], capture_output=True,
                         text=True, timeout=600)
    assert out.returncode == 0
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and "unavailable" in line


def test_reference_probe_decision(monkeypatch):
    bench = _load_bench()

    class Proc:
        def __init__(self, stdout):
            self.stdout, self.stderr, self.returncode = stdout, "", 0

    monkeypatch.delenv("DISABLE_MMA_V5", raising=False)
    tmem = '{"probe_error": "OutOfResources: out of resource: tensor memory, Required: 704, Hardware limit: 512"}\n'
    monkeypatch.setattr(bench.subprocess, "run", lambda *a, **k: Proc("log line\n" + tmem))
    assert "DISABLE_MMA_V5" in bench.probe_reference_backward(0)
    monkeypatch.setattr(bench.subprocess, "run", lambda *a, **k: Proc('{"probe_ok": true}\n'))
    assert bench.probe_reference_backward(0) == {}
    monkeypatch.setattr(bench.subprocess, "run", lambda *a, **k: Proc('{"probe_error": "ImportError: no triton"}\n'))
    assert bench.probe_reference_backward(0) == {}  # any other failure: leave the environment alone
    monkeypatch.setenv("DISABLE_MMA_V5", "1")
    assert bench.probe_reference_backward(0) == {}  # the user already chose


def test_dump_outputs_is_a_fixed_float32_sample_within_budget(tmp_path, monkeypatch):
    import numpy as np
    import torch

    bench = _load_bench()
    monkeypatch.setattr(bench, "DUMP_BYTES", 64 * 1024)
    out = torch.randn(1, 3000, 4, 8, dtype=torch.bfloat16)
    arrays = {"out": out, "dq": out * 2, "dk": torch.randn(1, 3000, 2, 8), "dv": torch.randn(1, 3000, 2, 8)}
    a = bench.dump_outputs(str(tmp_path / "a"), arrays, rank=1, world=2)
    bench.dump_outputs(str(tmp_path / "b"), arrays, rank=1, world=2)  # a second run writes the same files
    assert a["arrays"] == ["dk", "dq", "dv", "out"] and 0 < a["token_rows"] < 3000
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["dk_rank1.npy", "dq_rank1.npy", "dv_rank1.npy", "out_rank1.npy"]
    dumped = {f: np.load(tmp_path / "a" / f) for f in files}
    assert 2 * sum(x.nbytes for x in dumped.values()) <= 64 * 1024  # both ranks together fit the budget
    for f, x in dumped.items():
        assert x.dtype == np.float32 and x.shape[1] == a["token_rows"]
        assert np.array_equal(x, np.load(tmp_path / "b" / f))
    # every dumped row is a token row of the input, the same rows in every array
    full = out.float().numpy()[0]
    idx = [next(i for i in range(3000) if np.array_equal(r, full[i])) for r in dumped["out_rank1.npy"][0]]
    assert idx == sorted(set(idx))
    assert np.array_equal(dumped["dv_rank1.npy"][0], arrays["dv"].numpy()[0, idx])
    small = bench.dump_outputs(str(tmp_path / "c"), {"out": out[:, :10]}, rank=0, world=1)
    assert small["token_rows"] == 10
    assert np.array_equal(np.load(tmp_path / "c" / "out.npy"), out[:, :10].float().numpy())


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True,
                         text=True, timeout=600)
    assert out.returncode != 0 and "--steps" in out.stderr

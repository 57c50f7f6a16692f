"""bench.py's process-level contract, checked without a GPU: stdout carries the JSON line and nothing else, ranks other
than 0 of the reference arm exit quietly, and the product arm refuses to run without a CUDA device."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None, code=None):
    e = dict(os.environ)
    e.update(env or {})
    cmd = [sys.executable, "-c", code] if code else [sys.executable, os.path.join(ROOT, "bench.py"), *args]
    return subprocess.run(cmd, cwd=ROOT, env=e, capture_output=True, text=True, timeout=600)


def test_stdout_is_reserved_for_the_json_line():
    code = ("import os, sys, bench\n"
            "bench._claim_stdout()\n"
            "print('library chatter')\n"                      # Python-level print
            "os.write(1, b'NCCL version 2.28.9+cuda12.9\\n')\n"   # C-level write to file descriptor 1
            "bench.emit({'metric': 'm', 'value': 1.5})\n"
            "print('more chatter')\n")
    r = _run([], code=code)
    assert r.returncode == 0, r.stderr
    assert r.stdout.strip().splitlines() == ['{"metric": "m", "value": 1.5}']
    assert "NCCL version" in r.stderr and "library chatter" in r.stderr and "more chatter" in r.stderr


def test_reference_arm_runs_on_rank_zero_only():
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"], env={"RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout == ""


def test_dump_outputs_writes_loss_and_a_fixed_parameter_sample(tmp_path, monkeypatch):
    import numpy as np
    import torch
    import bench
    model = torch.nn.Sequential(torch.nn.Linear(4, 3), torch.nn.Linear(3, 2))
    model[0].bias.requires_grad_(False)
    trainable = torch.cat([p.detach().reshape(-1) for p in model.parameters() if p.requires_grad]).numpy()
    bench.dump_outputs(str(tmp_path / "all"), torch.tensor(1.5), model)
    loss = np.load(tmp_path / "all" / "loss.npy")
    assert loss.dtype == np.float32 and loss.shape == () and loss == 1.5
    np.testing.assert_array_equal(np.load(tmp_path / "all" / "params.npy"), trainable)   # small model: all, model order
    monkeypatch.setattr(bench, "DUMP_PARAM_SAMPLE", 7)
    runs = []
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), torch.tensor(1.5), model)
        runs.append(np.load(tmp_path / d / "params.npy"))
    assert runs[0].dtype == np.float32 and runs[0].shape == (7,)
    np.testing.assert_array_equal(runs[0], runs[1])                                      # same positions every run
    pos = [int(np.flatnonzero(trainable == v)[0]) for v in runs[0]]
    assert pos == sorted(pos)


def test_steps_must_be_positive_and_dump_needs_the_cuda_arm():
    r = _run(["--impl", "reference", "--steps", "0"])
    assert r.returncode != 0 and "--steps" in r.stderr
    r = _run(["--impl", "reference", "--steps", "1", "--dump-outputs", "unused"])
    assert r.returncode != 0 and "--dump-outputs" in r.stderr


def test_product_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    r = _run(["--steps", "1", "--warmup", "0"])
    assert r.returncode != 0 and r.stdout == ""
    assert "CUDA" in r.stderr

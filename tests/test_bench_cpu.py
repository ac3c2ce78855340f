"""bench.py's host side on the CPU: the reference arm (the one leg that runs without a GPU) prints the contract's JSON
line, the other ranks of a torchrun launch stay silent, and the product arm refuses to run without a CUDA device."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")


def _run(args, env_extra=None, timeout=600):
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    env.update(env_extra or {})
    return subprocess.run([sys.executable, BENCH] + args, capture_output=True, text=True, cwd=ROOT, env=env, timeout=timeout)


def _json_lines(stdout):
    return [json.loads(l) for l in stdout.splitlines() if l.strip().startswith("{")]


@pytest.fixture(scope="module")
def reference_line():
    # the reference's own shape (BASELINE.json configs[0]): small enough for a CPU test
    r = _run(["--impl", "reference", "--shape", "seoul", "--steps", "2", "--warmup", "1"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = _json_lines(r.stdout)
    assert len(lines) == 1, "the reference arm prints exactly one JSON line on stdout"
    return lines[0]


def test_reference_arm_prints_the_contract_line(reference_line):
    d = reference_line
    assert d["impl"] == "reference"
    assert d["metric"] == "ngcf_epoch_time_fwd_bwd_bpr" and d["unit"] == "s/epoch"
    assert d["higher_is_better"] is False and d["data"] == "synthetic" and d["dtype"] == "f32"
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["gpu_launches"] == 0
    assert d["vs_baseline"] is None                                  # BASELINE.json publishes no number for this metric
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["steps"] == cb["steps"] == 2 and d["warmup"] == 1                   # the steps it ran, no time budget
    assert d["e2e"] == {"value": d["value"], "unit": "s/epoch", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_both_arms_name_the_workload_the_same_way(reference_line):
    """The driver compares the two arms' `config` dicts: both are built from make_workload()'s description."""
    sys.path.insert(0, ROOT)
    argv, sys.argv = sys.argv, [sys.argv[0]]
    try:
        import bench
        from seoul_tourism_recommendation_ngcf_b200 import synth
    finally:
        sys.argv = argv
    assert set(reference_line["config"]) == {"workload", "steps_per_epoch"}
    n_user, n_item, n_edges, emb, K = synth.SHAPES["seoul"]
    w = reference_line["config"]["workload"]
    assert w.startswith("seoul-shaped") and f"{n_user} users / {n_item} items / {n_edges} interactions" in w
    assert f"emb {emb}, {K} layers, batch {bench.BATCH}" in w
    assert reference_line["config"]["steps_per_epoch"] == n_edges // bench.BATCH


def test_reference_arm_runs_on_rank_zero_only():
    r = _run(["--impl", "reference", "--shape", "seoul", "--steps", "1", "--warmup", "0", "--gpus", "2"],
             {"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}, timeout=120)
    assert r.returncode == 0 and _json_lines(r.stdout) == []


def test_device_generated_shapes_have_no_reference_run():
    r = _run(["--impl", "reference", "--shape", "pl-1b"], timeout=120)
    assert r.returncode == 0
    (d,) = _json_lines(r.stdout)
    assert d["impl"] == "reference" and "unavailable" in d


def test_bad_arguments_are_refused():
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        r = _run(args, timeout=120)
        assert r.returncode == 2 and _json_lines(r.stdout) == [], args


def test_dump_outputs_writes_the_loss_and_every_gradient(tmp_path, monkeypatch):
    import numpy as np
    import torch
    import bench
    torch.manual_seed(0)
    m = torch.nn.Sequential(torch.nn.Embedding(5000, 16), torch.nn.Linear(16, 8))
    loss = m(torch.randint(0, 5000, (64,))).square().sum()
    loss.backward()
    bench.dump_outputs(str(tmp_path / "full"), loss, m)
    names = {"loss.npy", "grad.0.weight.npy", "grad.1.weight.npy", "grad.1.bias.npy"}
    assert set(os.listdir(tmp_path / "full")) == names
    got = np.load(tmp_path / "full" / "loss.npy")
    assert got.dtype == np.float64 and got.tolist() == [float(loss)]
    for k, p in m.named_parameters():
        g = np.load(tmp_path / "full" / f"grad.{k}.npy")
        assert g.dtype == np.float32 and np.array_equal(g, p.grad.numpy()), k
    # past the size limit: a seeded sample of every gradient's rows, the same rows on every call
    monkeypatch.setattr(bench, "DUMP_BYTES", 64 << 10)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), loss, m)
    assert sum(np.load(tmp_path / "s1" / f).nbytes for f in names - {"loss.npy"}) <= 64 << 10
    for f in names:
        a, b = np.load(tmp_path / "s1" / f), np.load(tmp_path / "s2" / f)
        assert np.array_equal(a, b), f
    full = {r.tobytes() for r in np.load(tmp_path / "full" / "grad.0.weight.npy")}
    part = np.load(tmp_path / "s1" / "grad.0.weight.npy")
    assert 0 < len(part) < 5000 and all(r.tobytes() in full for r in part)


def test_product_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("this box has a GPU")
    r = _run(["--steps", "1", "--warmup", "1", "--no-cpu-baseline", "--no-epoch", "--no-extra"], timeout=300)
    assert r.returncode != 0 and _json_lines(r.stdout) == []
    assert "CUDA" in r.stderr

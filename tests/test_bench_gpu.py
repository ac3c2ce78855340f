"""bench.py on the GPU: --dump-outputs writes the loss and the parameter gradients of the last timed step, two runs with
the same arguments compute the same step (to the rounding of the gradients' float atomics), and --steps sets the number
of timed steps of every leg."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import seoul_tourism_recommendation_ngcf_b200 as pkg
from seoul_tourism_recommendation_ngcf_b200 import synth
from tests._golden import rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _env():
    return {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")}


def _bench(out_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1",
                        "--no-cpu-baseline", "--no-epoch", "--no-extra", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, cwd=ROOT, env=_env(), timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    (line,) = [json.loads(l) for l in r.stdout.splitlines() if l.strip().startswith("{")]
    return line


def test_dumped_outputs_are_the_same_on_every_run(tmp_path):
    lines = [_bench(tmp_path / d) for d in ("a", "b")]
    assert [d["steps"] for d in lines] == [2, 2]
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(os.listdir(tmp_path / "b"))
    n_user, n_item, _, emb, K = synth.SHAPES["gowalla"]
    want = {"loss.npy", "grad.user_embedding.weight.npy", "grad.item_embedding.weight.npy"}
    want |= {f"grad.w{w}_list.{k}.{p}.npy" for w in (1, 2) for k in range(K) for p in ("weight", "bias")}
    assert set(files) == want
    assert np.load(tmp_path / "a" / "grad.user_embedding.weight.npy").shape == (n_user, emb)
    assert np.load(tmp_path / "a" / "grad.item_embedding.weight.npy").shape == (n_item, emb)
    total = 0
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == (np.float64 if f == "loss.npy" else np.float32) and np.isfinite(a).all(), f
        assert np.abs(a).max() > 0, f
        assert rel_err(a, b) <= 1e-5, f
        total += a.nbytes
    assert total <= 64 << 20


def test_dump_is_the_last_timed_graph_replay_and_every_leg_runs_steps(tmp_path, monkeypatch, capsys):
    """In-process run of the default (graphed) path with the extra shapes: every GraphedStep call is recorded, so the
    dump can be matched with the call that produced it."""
    import bench
    steps, warm = 2, 3                                               # --warmup 1 runs bench's minimum of 3
    graphs, main = [], {}
    call = pkg.GraphedStep.__call__

    def recorded(self, batch):
        loss = call(self, batch)
        if not hasattr(self, "_test_serial"):
            self._test_serial = len(graphs)
            graphs.append({"optimizer": self.optimizer is not None, "losses": []})
        graphs[self._test_serial]["losses"].append(float(loss.detach()))
        if self._test_serial == 0 and len(graphs[0]["losses"]) == warm + steps:
            main["grads"] = {k: p.grad.detach().cpu().numpy().copy() for k, p in self.model.named_parameters()
                             if p.grad is not None}
        return loss

    dumps = []
    dump = bench.dump_outputs

    def recorded_dump(out_dir, loss, model):
        dumps.append([len(g["losses"]) for g in graphs])
        dump(out_dir, loss, model)

    monkeypatch.setattr(pkg.GraphedStep, "__call__", recorded)
    monkeypatch.setattr(bench, "dump_outputs", recorded_dump)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", str(steps), "--warmup", "1", "--no-cpu-baseline",
                                      "--no-epoch", "--dump-outputs", str(tmp_path)])
    bench.run_ours(bench.parse_args())
    (line,) = [json.loads(l) for l in capsys.readouterr().out.splitlines() if l.strip().startswith("{")]

    # one dump, right after the main graph's warm-up and timed replays, holding its last timed replay's outputs
    assert dumps == [[warm + steps]]
    assert not graphs[0]["optimizer"]
    assert np.load(tmp_path / "loss.npy").tolist() == [graphs[0]["losses"][warm + steps - 1]]
    assert set(os.listdir(tmp_path)) == {"loss.npy"} | {f"grad.{k}.npy" for k in main["grads"]}
    for k, g in main["grads"].items():
        assert np.array_equal(np.load(tmp_path / f"grad.{k}.npy"), g), k
    # the extra shapes: one graph each, 3 warm-up replays + --steps timed replays
    assert line["steps"] == steps and set(line["extra"]) == {"amazon-book", "yelp2018", "seoul"}
    assert all(v["steps"] == steps for v in line["extra"].values()), line["extra"]
    extra = [g for g in graphs[1:] if not g["optimizer"]]
    assert [len(g["losses"]) for g in extra] == [3 + steps] * 3


def test_device_generated_shape_runs_steps_and_dumps_its_last_timed_step(tmp_path):
    """pl-10m with more steps than the old cap of 10: the dump comes after 3 warm-up + --steps replays and holds the
    loss of the last of them."""
    steps = 12
    code = f"""
import sys
sys.argv = ["bench.py", "--shape", "pl-10m", "--steps", "{steps}", "--warmup", "1", "--dump-outputs", {str(tmp_path)!r}]
import bench
import seoul_tourism_recommendation_ngcf_b200 as pkg
losses = []
call = pkg.GraphedStep.__call__
def recorded(self, batch):
    loss = call(self, batch)
    losses.append(float(loss.detach()))
    return loss
pkg.GraphedStep.__call__ = recorded
dump = bench.dump_outputs
def recorded_dump(out_dir, loss, model):
    print("DUMP", len(losses), repr(losses[-1]), file=sys.stderr, flush=True)
    dump(out_dir, loss, model)
bench.dump_outputs = recorded_dump
args = bench.parse_args()
bench.protect_stdout()
bench.run_pl(args)
"""
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, env=_env(), timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    (line,) = [json.loads(l) for l in r.stdout.splitlines() if l.strip().startswith("{")]
    assert line["steps"] == steps
    (dump,) = [l.split() for l in r.stderr.splitlines() if l.startswith("DUMP ")]
    assert int(dump[1]) == 3 + steps
    assert np.load(tmp_path / "loss.npy").tolist() == [float(dump[2])]
    n_user, n_item, _, emb, _ = synth.SHAPES["pl-10m"]
    assert np.load(tmp_path / "grad.user_embedding.weight.npy").shape == (n_user, emb)
    assert np.load(tmp_path / "grad.item_embedding.weight.npy").shape == (n_item, emb)

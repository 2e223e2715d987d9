"""`bench.py --impl reference` contract: the reference cannot run here (it needs OneFlow) → one JSON line saying so, rc 0."""
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_reports_unavailable():
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--gpus", "1", "--steps", "2", "--warmup", "3"],
                       cwd=REPO, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-500:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference"
    assert "unavailable" in line or "value" in line      # (a value only if OneFlow were importable)


def test_bench_rejects_zero_steps():
    r = subprocess.run([sys.executable, "bench.py", "--steps", "0"], cwd=REPO, capture_output=True, text=True, timeout=300)
    assert r.returncode == 2 and "--steps" in r.stderr


def test_dump_outputs_writes_a_seeded_float32_sample(tmp_path):
    """`bench.py --dump-outputs`: the loss dict and the same sample of the model state on every call."""
    import numpy as np
    import torch

    sys.path.insert(0, REPO)
    import bench

    torch.manual_seed(0)
    model = torch.nn.Sequential(torch.nn.Linear(100, 100), torch.nn.LayerNorm(100)).bfloat16()
    model.register_buffer("steps", torch.tensor(3))          # integer state is not sampled
    loss = {"lm_loss": torch.tensor(2.5)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), loss, model)
    assert sorted(os.listdir(tmp_path / "a")) == ["lm_loss.npy", "state_sample.npy"]
    a, b = np.load(tmp_path / "a" / "state_sample.npy"), np.load(tmp_path / "b" / "state_sample.npy")
    assert a.dtype == np.float32 and a.shape == (bench.DUMP_SAMPLES_PER_TENSOR + 3 * 100,) and np.array_equal(a, b)
    w = model[0].weight.detach().float().flatten().numpy()
    assert np.isin(a[:bench.DUMP_SAMPLES_PER_TENSOR], w).all()              # sampled from the large tensor
    assert np.array_equal(a[bench.DUMP_SAMPLES_PER_TENSOR:][:100], model[0].bias.detach().float().numpy())   # small: whole
    assert np.load(tmp_path / "a" / "lm_loss.npy") == np.float32(2.5)


_WATCHDOG_SCRIPT = r"""
import json, os, sys, time
sys.path.insert(0, {repo!r})
os.environ["MASTER_PORT"] = "{port}"
import bench

role = sys.argv[1]
layouts = {{"dp2": {{"value": 1.0}}}}


def emit():
    print(json.dumps({{"value": 1.0, "layouts": layouts}}), flush=True)


w = bench._ExtrasWatchdog(2, emit, layouts, limit_s=float(sys.argv[2]))
w.begin("tp2")
if role == "fails":
    w.fail("tp2", "RuntimeError: boom")          # must not return
    print("NOT REACHED")
elif role == "peer":
    time.sleep(30)                                # "blocked in a collective": the poller has to end the process
    print("NOT REACHED")
"""


def _run_watchdog(tmp_path, role, limit, flag_first=False):
    script = tmp_path / f"wd_{role}.py"
    script.write_text(_WATCHDOG_SCRIPT.format(repo=REPO, port=40000 + os.getpid() % 20000))
    return subprocess.Popen([sys.executable, str(script), role, str(limit)], cwd=REPO, stdout=subprocess.PIPE,
                            stderr=subprocess.PIPE, text=True)


def test_extras_watchdog_keeps_the_headline_line(tmp_path):
    """A failure (or a hang) inside an extra layout must end every rank with exit code 0 and the JSON line printed by
    whoever calls ``emit`` (rank 0 in bench.py): the failing rank raises the flag, the peers' pollers see it."""
    # same parent process => same flag file for both "ranks"
    peer = _run_watchdog(tmp_path, "peer", 60)
    failing = _run_watchdog(tmp_path, "fails", 60)
    out_f, _ = failing.communicate(timeout=60)
    out_p, _ = peer.communicate(timeout=60)
    assert failing.returncode == 0 and peer.returncode == 0
    for out in (out_f, out_p):
        assert "NOT REACHED" not in out
        line = json.loads(out.strip().splitlines()[-1])
        assert line["value"] == 1.0 and "boom" in line["layouts"]["tp2"]["error"]
    flag = os.path.join("/tmp", f"libai_b200_bench_fail_{40000 + os.getpid() % 20000}_{os.getpid()}")
    if os.path.exists(flag):
        os.remove(flag)
    # a layout that exceeds its time limit ends the same way
    slow = _run_watchdog(tmp_path, "peer", 1.0)
    out_s, _ = slow.communicate(timeout=60)
    assert slow.returncode == 0 and "exceeded" in json.loads(out_s.strip().splitlines()[-1])["layouts"]["tp2"]["error"]
    if os.path.exists(flag):
        os.remove(flag)

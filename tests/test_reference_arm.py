"""The reference arm of bench.py (baseline/reference_arm.py + baseline/shims): the UNMODIFIED reference runs its own local
training path on stand-ins for its external dependencies.  These tests pin down what the stand-ins promise."""
import hashlib
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE = os.path.join(ROOT, "baseline")
ORACLE = os.path.join(ROOT, "oracle")
REF = os.path.join(ORACLE, "_ref")
# sha256 of the original project's files, taken from its checkout (tests/golden/reference_sha256.txt)
GOLDEN_SHA256 = os.path.join(ROOT, "tests", "golden", "reference_sha256.txt")

needs_ref = pytest.mark.skipif(not os.path.exists(os.path.join(REF, "SHA256SUMS")),
                               reason="the original project is not installed under oracle/_ref (build() found no checkout of it)")


def test_standins_do_not_import_the_product():
    """Nothing under baseline/shims (nor the harness) may pull in this repo's package: the reference arm must not run on any
    of the product's models, kernels or engine."""
    bad = []
    for dirpath, _, files in os.walk(os.path.join(BASE, "shims")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                if "colearn_federated_learning_b200" in src.replace("``colearn_federated_learning_b200``", ""):
                    bad.append(os.path.join(dirpath, f))
    assert not bad, bad
    harness = open(os.path.join(BASE, "reference_arm.py")).read()
    assert "import colearn_federated_learning_b200" not in harness and "from colearn_federated_learning_b200" not in harness


@needs_ref
def test_installed_reference_is_byte_identical():
    sys.path.insert(0, ORACLE)
    try:
        import install_ref
        sums = install_ref.verify(REF)
    finally:
        sys.path.remove(ORACLE)
    assert {"federated_coordinator.py", "client_federated.py", "datasets.py", "event_parser.py", "settings.py"} <= set(sums)
    golden = dict(reversed(line.split()) for line in open(GOLDEN_SHA256) if line.strip())
    assert set(sums) == set(golden)
    for rel, h in sums.items():
        assert hashlib.sha256(open(os.path.join(REF, rel), "rb").read()).hexdigest() == h == golden[rel], rel


@needs_ref
def test_reference_arm_runs_the_reference_local_training():
    """`bench.py --impl reference` end to end on a small CSV: one JSON line, the reference's own modules on the path, no
    product module loaded, a finite checkpoint."""
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1",
                        "--samples", "96"], capture_output=True, text=True, timeout=600, cwd=ROOT,
                       env={**os.environ, "CUDA_VISIBLE_DEVICES": ""})
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, p.stdout
    rec = json.loads(lines[0])
    assert rec["impl"] == "reference" and "unavailable" not in rec
    assert rec["config"]["workers"] == 2 and rec["config"]["samples_per_worker"] == 48 and rec["config"]["checkpoint_finite"]
    assert rec["reference"]["product_modules_loaded"] == [] and rec["reference"]["unmodified"]
    assert rec["value"] > 0 and rec["e2e"]["value"] > 0


def test_standin_semantics():
    """send/get move a module in place, federate = contiguous ceil(N/K) shards, the loader goes worker by worker, and
    federated_avg is the unweighted mean accumulated into the first model (PySyft 0.2 semantics the reference relies on)."""
    code = r"""
import sys, math
sys.path.insert(0, sys.argv[1])
import torch, syft as sy
from torch import nn
from torch.utils.data import TensorDataset
from syft.frameworks.torch.fl import utils
hook = sy.TorchHook(torch)
a, b = sy.VirtualWorker(hook, "a"), sy.VirtualWorker(hook, "b")
assert set(hook.local_worker._known_workers) == {"me", "a", "b"}
ds = TensorDataset(torch.arange(10.).view(10, 1), torch.arange(10.).view(10, 1))
fed = ds.federate((a, b))
assert fed.workers == ["a", "b"] and len(fed["a"]) == 5 and len(fed["b"]) == 5
assert fed["a"].data.view(-1).tolist() == [0, 1, 2, 3, 4]
loader = sy.FederatedDataLoader(fed, batch_size=1, shuffle=True)
seen = [(d.location.id, float(d)) for d, t in loader]
assert len(loader) == 10 and [w for w, _ in seen] == ["a"] * 5 + ["b"] * 5
assert sorted(v for w, v in seen if w == "a") == [0, 1, 2, 3, 4]
m = nn.Linear(2, 1)
assert m.send(a) is m and m.location is a and m.get() is m
m1, m2 = nn.Linear(2, 1), nn.Linear(2, 1)
w1, w2 = m1.weight.detach().clone(), m2.weight.detach().clone()
avg = utils.federated_avg({"a": m1, "b": m2})
assert avg is m1 and torch.allclose(m1.weight, (w1 + w2) / 2)
x = torch.ones(3).send(a)
assert x.location is a and x.get() is x
print("OK")
"""
    p = subprocess.run([sys.executable, "-c", code, os.path.join(BASE, "shims")], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0 and "OK" in p.stdout, p.stderr[-2000:]


def test_bench_ref_local_data_matches_the_reference_arms_csv(tmp_path):
    """Both arms train on the same rows: the CSV generator of the reference arm, read through this repo's dataset class,
    gives MinMax-scaled features in [0, 1] and the binary attack label."""
    sys.path.insert(0, ROOT)
    try:
        import bench
        x0, y0 = bench.load_ref_local_data(64, 0, 2)
        x1, y1 = bench.load_ref_local_data(64, 1, 2)
    finally:
        sys.path.remove(ROOT)
    assert x0.shape == (32, 10) and x1.shape == (32, 10) and y0.shape == (32, 1)
    x = torch.cat([x0, x1])
    assert float(x.min()) == 0.0 and float(x.max()) == 1.0 and set(torch.cat([y0, y1]).view(-1).tolist()) <= {0.0, 1.0}


def test_bench_stdout_carries_the_result_line_only():
    """bench.py points file descriptor 1 at stderr for the life of the process (NCCL prints its version banner to fd 1 at
    world > 1) and keeps Python's stdout for the one JSON line of the contract."""
    # a library-style write to fd 1 from inside the process (here: at exit, after bench.py has re-pointed the descriptor)
    # must land on stderr, not next to the result line
    probe = ("import os, sys, json, runpy, atexit\n"
             "atexit.register(lambda: os.write(1, b'banner from a C library\\n'))\n"
             "sys.argv = ['bench.py', '--gpus', '1']\n"
             "runpy.run_path(%r, run_name='__main__')\n" % os.path.join(ROOT, "bench.py"))
    p = subprocess.run([sys.executable, "-c", probe], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, p.stdout
    assert "unavailable" in json.loads(lines[0]) or "value" in json.loads(lines[0])
    assert "banner from a C library" in p.stderr

"""``bench.py --impl reference``: the UNMODIFIED reference (``oracle/_ref``, byte-identical copy of the original project,
sha256-checked) running its own stock local-training path on this box.

    events "(ip, TRAINING)" -> Coordinator.on_message (reference parser, registry, VirtualWorker per device)
      -> the window timer's callback = starting_training_local (fc.py:318-392)
           NetworkTrafficDataset(csv).federate(workers) -> FederatedDataLoader(batch 1, shuffle)
           for every worker: cf.train_local (cf.py:82-127: send, zero_grad, forward, SSE, backward, SGD step, get)
           utils.federated_avg -> torch.save(test.pth)

One step = one such training = one federated round over N workers (N = ``--gpus``; the reference's local mode trains its
workers one after the other in one process — that IS its stock behaviour — so ranks > 0 have nothing to do).  The
reference's external dependencies ``syft`` / ``paho`` do not exist offline; ``baseline/shims`` holds builder-written
plain-PyTorch stand-ins for those external names only (see its README: semantics kept, PySyft's per-op serialisation
cost NOT reproduced, so the reference runs faster here than it would with the real PySyft).

Only the wait of the temporal window (``Timer(window, fn)``, 1 s by default) is taken out of the timed region: the
module-global ``Timer`` name of the reference is pointed at a class that records the callback, and the harness calls it.

Nothing in this file (or the shims) imports ``colearn_federated_learning_b200``.
"""
from __future__ import annotations

import io
import json
import os
import sys
import tempfile
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
ORACLE = os.path.join(ROOT, "oracle")
REF = os.path.join(ORACLE, "_ref")
SHIMS = os.path.join(HERE, "shims")

PUBLISHED_ROUNDS_PER_S = 0.1133     # BASELINE.md: 12 rounds x 1000 it, 2 x RPi 3B+
CSV_HEADER = ["pkSeqID", "proto", "saddr", "sport", "daddr", "dport", "seq", "stddev", "N_IN_Conn_P_SrcIP", "min", "state_number",
              "mean", "N_IN_Conn_P_DstIP", "drate", "srate", "max", "attack", "category", "subcategory"]
FEATURES = ["seq", "stddev", "N_IN_Conn_P_SrcIP", "min", "state_number", "mean", "N_IN_Conn_P_DstIP", "drate", "srate", "max"]


def write_synthetic_csv(path: str, n: int, seed: int = 0) -> None:
    """``n`` rows in the Bot-IoT "10-best" layout (the reference's ``dataset_example`` header): 10 numeric features, a
    binary ``attack`` label that is a noisy linear function of them, the remaining columns filled with plausible
    constants.  numpy/pandas only — both bench arms read this same file."""
    import numpy as np
    import pandas as pd

    rng = np.random.default_rng(seed)
    x = rng.random((n, 10))
    w = np.array([1.5, -2.0, 1.0, 0.5, -1.0, 2.0, -1.5, 1.0, -0.5, 1.0])
    y = ((x - 0.5) @ w + 0.1 * rng.standard_normal(n) > 0).astype(np.int64)
    scale = np.array([262144.0, 2.5, 100.0, 5.0, 6.0, 5.0, 100.0, 1.0, 1.0, 5.0])
    df = pd.DataFrame({c: 0 for c in CSV_HEADER}, index=range(n))
    df["pkSeqID"] = np.arange(1, n + 1)
    df["proto"], df["saddr"], df["daddr"] = "udp", "192.168.100.150", "192.168.100.3"
    df["sport"], df["dport"] = 6551, 80
    for j, c in enumerate(FEATURES):
        df[c] = np.round(x[:, j] * scale[j], 6)
    df["attack"] = y
    df["category"] = np.where(y == 1, "DDoS", "Normal")
    df["subcategory"] = np.where(y == 1, "UDP", "Normal")
    df[CSV_HEADER].to_csv(path, index=False)


class _CapturedTimer:
    """Stands in for ``threading.Timer`` inside the reference module: records (interval, function); ``start`` does nothing."""
    last = None

    def __init__(self, interval, function, args=None, kwargs=None):
        self.interval, self.function = interval, function
        self.args, self.kwargs = args or (), kwargs or {}
        _CapturedTimer.last = self

    def start(self):
        pass

    def cancel(self):
        pass

    def fire(self):
        return self.function(*self.args, **self.kwargs)


def unavailable(why: str) -> None:
    if int(os.environ.get("RANK", "0")) == 0:
        print(json.dumps({"impl": "reference", "unavailable": why}))


def main(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return          # the reference's local mode is one process training its workers sequentially
    try:
        sys.path.insert(0, ORACLE)
        import install_ref
        sums = install_ref.verify(REF)
    except Exception as exc:  # noqa: BLE001
        unavailable(f"oracle/_ref is not installed ({exc}); run `python oracle/install_ref.py --src <checkout of the original project>`")
        return
    # the reference's flat modules + the stand-ins first on the path; the product's repo root off it
    sys.path[:] = [REF, SHIMS] + [p for p in sys.path if os.path.abspath(p or ".") not in (ROOT, HERE, ORACLE)]

    import torch

    total = args.samples or 8192
    n_workers = max(1, world if world > 1 else args.gpus)
    K, W = max(1, args.steps), max(3, args.warmup)
    use_cuda = torch.cuda.is_available()

    sink = io.StringIO()
    real_stdout = sys.stdout
    sys.stdout = sink                      # train_local prints a progress line every 30 batches
    try:
        import federated_coordinator as fc   # the reference's module (oracle/_ref)
        import settings as ref_settings
        import paho.mqtt.client as mqtt

        assert os.path.dirname(os.path.abspath(fc.__file__)) == REF
        fc.Timer = _CapturedTimer
        with tempfile.TemporaryDirectory() as tmp:
            csv = os.path.join(tmp, "synthetic_unsw.csv")
            write_synthetic_csv(csv, total, seed=0)
            coord = fc.Coordinator(window=1, remote=False, federated_round=1, encryption=False, iot_validation=False)
            coord.path = os.path.join(tmp, "test.pth")
            coord.args.test_path = csv
            coord.args.lr = args.lr
            topic = "topic/state"
            coord.connect("localhost", 1883)
            coord.subscribe(topic, qos=0)
            pub = mqtt.Client("devices")
            pub.connect("localhost")

            def one_training():
                if os.path.exists(coord.path):
                    os.remove(coord.path)       # every timed training starts like the README demo: no checkpoint yet
                _CapturedTimer.last = None
                if use_cuda:
                    torch.cuda.synchronize()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                t0 = time.perf_counter()
                for i in range(n_workers):
                    pub.publish(topic, f"(192.168.1.{7 + i}, TRAINING)")
                timer = _CapturedTimer.last
                assert timer is not None and len(ref_settings.training_devices) == n_workers
                timer.fire()                    # = starting_training_local(lower, upper, path, args, server)
                if use_cuda:
                    e1.record()
                    torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                assert os.path.exists(coord.path) and len(ref_settings.training_devices) == 0 and ref_settings.event_served == 0
                sink.seek(0)
                sink.truncate()
                return dt, (e0.elapsed_time(e1) if use_cuda else dt * 1e3)

            for _ in range(W):
                one_training()
            wall, dev_ms = 0.0, 0.0
            for _ in range(K):
                dt, ms = one_training()
                wall += dt
                dev_ms += ms
            state = torch.load(coord.path, map_location="cpu")
            finite = all(bool(torch.isfinite(v).all()) for v in state.values())
            n_params = sum(v.numel() for v in state.values())
    finally:
        sys.stdout = real_stdout

    product_loaded = sorted(m for m in sys.modules if m.startswith("colearn_federated_learning_b200"))
    per_worker = -(-total // n_workers)
    value = K / (dev_ms * 1e-3)
    out = {
        "impl": "reference",
        "metric": "FL rounds/sec (whole box, device-timed, max over ranks)",
        "value": value, "unit": "rounds/s", "n_gpus": world if world > 1 else args.gpus, "steps": K, "warmup": W,
        "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": value / PUBLISHED_ROUNDS_PER_S, "dtype": "fp32",
        "data": "synthetic UNSW-IoT-shaped CSV (Bot-IoT 10-best header) / random-init weights",
        "config": {"name": "ref_local", "model": "ffnn", "description": "reference local (VirtualWorker) training, fc.py:318-392: FFNN 10-50-30-10-1, "
                   "sum-squared-error, batch 1, SGD lr 0.01, 1 local epoch over a fixed CSV split into N contiguous shards, uniform FedAvg, test.pth",
                   "global_batch": 1, "batch_size_per_worker": 1, "seq_len": None, "parallelism": f"fedavg sequential x{n_workers} (one process)",
                   "total_samples": total, "samples_per_worker": per_worker, "workers": n_workers, "local_epochs": 1,
                   "local_sgd_steps_per_round": per_worker, "lr": args.lr, "loss": "sse",
                   "device": "cuda:0" if use_cuda else "cpu", "gpus_used": 1 if use_cuda else 0,
                   "params": n_params, "checkpoint_finite": finite,
                   "timed_region": "events -> on_message -> starting_training_local (CSV read, MinMax, federate, K x train_local, federated_avg, save); "
                                   "the window wait itself (Timer, 1 s default) is excluded",
                   "l2": "inputs re-read from the CSV and re-uploaded sample by sample every round (reference behaviour)",
                   "baseline_ref": "0.1133 rounds/s = 12 rounds x 1000 it on 2x RPi 3B+ (BASELINE.md)"},
        "e2e": {"value": K / wall, "unit": "rounds/s",
                # ToTensor uploads every sample and label separately (datasets.py:63-69); the progress line reads the loss back every 30 batches
                "h2d_bytes_per_step": int(total * 11 * 4) if use_cuda else 0,
                "d2h_bytes_per_step": int((n_workers * ((per_worker * n_workers + 29) // 30)) * 4 + n_params * 4) if use_cuda else 0,
                "timing": "host clock around the same region"},
        "gpu_launches": 0,
        "kernels": "ATen / cuBLAS only (stock torch ops issued by the reference's Python loop)",
        "reference": {"path": "oracle/_ref", "sha256": sums, "unmodified": True,
                      "entry": "federated_coordinator.Coordinator.on_message -> starting_training_local -> client_federated.train_local",
                      "module_patches": ["federated_coordinator.Timer -> records the callback so the harness can skip the window wait"],
                      "standins": "baseline/shims/{syft,paho}: BUILDER-WRITTEN plain-PyTorch stand-ins for the reference's external, "
                                  "offline-unavailable dependencies (PySyft 0.2.x, paho-mqtt); PySyft's per-op cost is not reproduced, "
                                  "so this arm is faster than the reference with its real dependencies would be",
                      "product_modules_loaded": product_loaded},
    }
    print(json.dumps(out))

#!/usr/bin/env python
"""Headline benchmark: FL rounds/sec on N GPUs of one box (BASELINE.json metric).

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29511 bench.py --gpus 8 --steps 20 --warmup 3

One **step = one federated round**: broadcast θ from the coordinator (rank 0) to the selected
workers → each worker runs its local epoch(s) of SGD (forward, loss, backward, optimizer step —
nothing skipped) on its private shard → FedAvg weighted reduce → server apply.  Default config is
BASELINE.json config 2 (``mlp`` 10→64→64→2, batch 1 like the reference's ``Arguments``, 1 local
epoch, sample-count-weighted FedAvg) with a FIXED total dataset that ``federate()`` splits into N
contiguous shards (reference ``dataset.federate(workers)``, fc.py:347-350) — i.e. strong scaling.

Timing: W untimed warm-up rounds, then K rounds each bracketed by CUDA events on the launching
stream with an (untimed) L2 flush in between, barrier + synchronize on both sides of the region,
MAX over ranks.  ``e2e`` re-measures through the same public API (``FederatedEngine.run_rounds``)
with, every round, the H2D copy of the round's shard from pinned host memory and a D2H read of
the round's loss, timed by the host clock.  ``--impl reference`` reports that the reference
cannot be installed offline (DESIGN.md); ``--impl torch_nccl`` runs the stock-PyTorch + NCCL
comparator from ``baseline/`` for the same metric/config.

Other ``--config`` values: ``cfg3`` / ``cfg4`` / ``cfg5`` / ``ffnn`` (the remaining BASELINE configs on the GPU engine) and
four host-clocked end-to-end runs of the reference's own published experiments through the classic control plane, which
also run on a box without a GPU: ``cfg1`` (VirtualWorker mode), ``paper`` (12 rounds x 1000 it, 2 remote worker
processes over TCP — paper Table 1), ``fulldata`` (733 672 samples on one remote worker) and ``smpc`` (the encrypted demo).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

PUBLISHED_ROUNDS_PER_S = 0.1133  # BASELINE.md: 12 rounds x 1000 it, 2x RPi 3B+ (best published rounds/s)

CONFIGS = {
    # name: (model, total_samples, batch, local_epochs, select_k, description)
    "paper": ("ffnn", 2000, 1, 1, None, "the reference's published experiment (paper Table 1 / BASELINE.md headline): FFNN 10-50-30-10-1, BCE, "
                                        "batch 1, 12 rounds x 1000 local iterations, 2 remote workers over TCP, coordinator + remote_worker.py CLIs' code path"),
    "fulldata": ("ffnn", 733672, 1, 1, None, "the reference's full-dataset run (BASELINE.md: 733 672 samples, batch 1, 1 round, 1 remote worker: "
                                             "4 481.6 s = 163.7 SGD steps/s on an RPi 3B+)"),
    "smpc": ("ffnn", 1000, 1, 1, None, "the reference's SMPC demo (paper Fig. 7): encrypted training of the FFNN on 1000 secret-shared items, "
                                       "2 workers + crypto provider (federated_coordinator.py -e code path)"),
    "ref_local": ("ffnn", 8192, 1, 1, None, "the reference's local (VirtualWorker) training, fc.py:318-392, with one worker per GPU: FFNN 10-50-30-10-1 "
                                            "(the reference's production model), sum-squared-error, batch 1, SGD lr 0.01, 1 local epoch over a fixed "
                                            "8192-row CSV split into N contiguous shards, uniform FedAvg — the SAME config `--impl reference` runs"),
    "cfg1": ("mlp", 2048, 1, 1, None, "federated_coordinator.py VirtualWorker mode, 2 workers, 10-feature MLP, 1 round (BASELINE config 1, plumbing)"),
    "cfg2": ("mlp", 8192, 1, 1, None, "3-layer MLP 10-64-64-2, 1 local epoch, all workers (BASELINE config 2)"),
    "cfg3": ("mlp", 8192, 1, 5, 4, "same MLP, 5 local epochs, temporal window selects 4 of 8 (BASELINE config 3)"),
    "ffnn": ("ffnn", 8192, 1, 1, None, "reference FFNN 10-50-30-10-1, BCE, 1 local epoch"),
    "cfg4": ("resnet18", 2048, 128, 1, None, "ResNet-18 bf16 on synthetic 32x32 images (BASELINE config 4)"),
    "cfg5": ("wide_mlp", 8192, 1024, 1, None, "wide MLP 10-4096x4-2 bandwidth sweep (BASELINE config 5)"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch_nccl"])
    ap.add_argument("--config", default=None, choices=sorted(CONFIGS),
                    help="default: ref_local (the config the reference arm runs) with BASELINE config 2 attached")
    ap.add_argument("--samples", type=int, default=None, help="total samples across all workers (strong scaling)")
    ap.add_argument("--batch-size", type=int, default=None)
    ap.add_argument("--local-epochs", type=int, default=None)
    ap.add_argument("--lr", type=float, default=0.01)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--nvlink-counters", action="store_true",
                    help="after the timed region, run the K rounds once more between two reads of this GPU's NVLink payload counters "
                         "(NVML) and report bytes per round next to the algorithmic count (config.nvlink)")
    ap.add_argument("--no-flush", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed rounds, write what the last timed round returned (global model, per-worker losses) "
                         "as DIR/<config>_<name>.npy (float32), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config in ("cfg1", "paper", "fulldata", "smpc")):
        ap.error("--dump-outputs covers the GPU engine configs of --impl ours (ref_local, cfg2, cfg3, ffnn, cfg4, cfg5)")
    return args


DUMP_MAX_ARRAYS = 4                      # the default line dumps two configs x (theta, losses)
DUMP_MAX_ELEMS = 64 * 1024 * 1024 // 4 // DUMP_MAX_ARRAYS   # 64 MB of float32 in all


def dump_outputs(out_dir: str, prefix: str, arrays) -> None:
    """``out_dir/<prefix>_<name>.npy`` in float32 for every tensor of ``arrays``.  An array of more than
    ``DUMP_MAX_ELEMS`` elements is stored as a sample: the elements at sorted indices drawn by a generator seeded 0
    (the same indices every run), flattened."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        if t is None:
            continue
        flat = t.detach().float().cpu().reshape(-1)
        if flat.numel() > DUMP_MAX_ELEMS:
            idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ELEMS].sort().values
            arr = flat[idx].numpy()
        else:
            arr = t.detach().float().cpu().numpy()
        np.save(os.path.join(out_dir, f"{prefix}_{name}.npy"), arr)


def make_data(model: str, total: int, rank: int, world: int, seed: int = 0):
    import torch
    from colearn_federated_learning_b200.data import shard_bounds, synthetic_images, synthetic_unsw

    if model == "resnet18":
        x, y = synthetic_images(total, seed=seed)
        y = y.float().view(-1, 1)
    else:
        x, y = synthetic_unsw(total, seed=seed)
    lo, hi = shard_bounds(total, world)[rank]
    return x[lo:hi].contiguous(), y[lo:hi].contiguous()


def bench_cfg1(args) -> None:
    """BASELINE config 1: the whole classic control plane — events on the in-process bus, parser, registry, temporal
    window, selection, two VirtualWorkers training their contiguous shards (ONE persistent-kernel launch for both on a
    GPU, the PyTorch reference ops on a CPU-only box), FedAvg, ``test.pth`` — timed per training window on the host
    clock.  It is a plumbing configuration: what it measures is the framework overhead around a tiny fit."""
    import tempfile
    import time

    import torch

    from colearn_federated_learning_b200.control.arguments import Arguments
    from colearn_federated_learning_b200.control.bus import BusClient, InProcessBroker
    from colearn_federated_learning_b200.control.coordinator import Coordinator
    from colearn_federated_learning_b200.control.window import FakeClock

    model, total, bsz, epochs, _, desc = CONFIGS["cfg1"]
    total = args.samples or total
    device = torch.device("cuda", 0) if torch.cuda.is_available() else torch.device("cpu")
    a = Arguments()
    a.model, a.synthetic, a.batch_size, a.epochs, a.lr, a.loss = model, total, args.batch_size or bsz, args.local_epochs or epochs, args.lr, "xent"
    K, W = args.steps, max(3, args.warmup)
    with tempfile.TemporaryDirectory() as tmp:
        broker, clock = InProcessBroker(), FakeClock()
        c = Coordinator(1, False, 1, False, False, args=a, broker=broker, timer_factory=clock, path=os.path.join(tmp, "test.pth"),
                        device=device)
        c.connect()
        c.subscribe("topic/state")
        pub = BusClient("devices", broker=broker)
        pub.connect()

        def one_window():
            pub.publish("topic/state", "(192.168.1.7, TRAINING)")
            pub.publish("topic/state", "(192.168.1.8, TRAINING)")
            c.drain()
            clock.advance(1.0)          # the window closes: select, federate, train, FedAvg, save, deregister
            if device.type == "cuda":
                torch.cuda.synchronize()

        for _ in range(W):
            one_window()
        t0 = time.perf_counter()
        for _ in range(K):
            one_window()
        dt = time.perf_counter() - t0
        assert c.trainings_done == W + K
    value = K / dt
    print(json.dumps({
        "metric": "FL rounds/sec (classic coordinator, VirtualWorker mode, host clock)", "value": value, "unit": "rounds/s",
        "n_gpus": 1 if device.type == "cuda" else 0, "steps": K, "warmup": W, "ms_per_step": dt / K * 1e3, "higher_is_better": True,
        "scaling": "n/a", "vs_baseline": value / PUBLISHED_ROUNDS_PER_S, "dtype": "fp32",
        "data": "synthetic UNSW-IoT-shaped features / checkpoint carried from window to window", "impl": "ours",
        "config": {"name": "cfg1", "model": model, "description": desc, "workers": 2, "total_samples": total,
                   "local_sgd_steps_per_round": total // 2, "device": str(device),
                   "includes": "bus + parser + window + selection + federate + local SGD + FedAvg + atomic .pth save + reload"},
        "e2e": {"value": value, "unit": "rounds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "timing": "the measurement is already end to end (host clock around whole training windows)"},
        # per window on a GPU: 2 permutation kernels, 1 persistent-MLP launch (both workers), 1 fedavg_apply
        "gpu_launches": (4 * K) if device.type == "cuda" else 0}))


def bench_paper(args) -> None:
    """The experiment behind the reference's headline number (paper Table 1; BASELINE.md: 12 rounds x 1000 it on 2 x
    RPi 3B+ = 105.9 s, 0.1133 rounds/s): the real remote mode — two ``remote_worker.py`` PROCESSES hosting private
    shards and serving fit RPCs over TCP, the real ``Coordinator`` (MQTT-framed TCP bus, parser, registry, temporal
    window, ``training_remote``: per round ship theta, 1000 batch-1 SGD steps with BCE on every worker, FedAvg),
    checkpoint at the end.  One step = one whole training (12 rounds); the value is rounds/s like the paper's.
    Runs wherever the workers run: on a GPU box they train through the persistent kernel, on a CPU-only box through
    the native host executor."""
    import subprocess
    import tempfile

    import torch

    from colearn_federated_learning_b200.control.arguments import Arguments
    from colearn_federated_learning_b200.control.bus import BusClient, TcpBroker
    from colearn_federated_learning_b200.control.coordinator import Coordinator
    from colearn_federated_learning_b200.control.window import FakeClock

    full = args.config == "fulldata"
    model, total, bsz, epochs, _, desc = CONFIGS[args.config]
    rounds, n_workers = (1, 1) if full else (12, 2)
    per_worker = (args.samples or total) // n_workers
    K, W = max(1, args.steps), max(3, args.warmup)
    use_cuda = torch.cuda.is_available()
    topic = "topic/state"
    procs = []
    with tempfile.TemporaryDirectory() as tmp:
        broker = TcpBroker("127.0.0.1", 0).start()
        try:
            ports = []
            for i in range(n_workers):
                import socket
                with socket.socket() as sk:
                    sk.bind(("127.0.0.1", 0))
                    ports.append(sk.getsockname()[1])
            for i, port in enumerate(ports):
                cmd = [sys.executable, os.path.join(ROOT, "remote_worker.py"), "--host", "127.0.0.1", "-p", str(port), "-b", "127.0.0.1",
                       "--broker-port", str(broker.port), "-t", topic, "-w", "0.2", "--synthetic", str(per_worker), "--seed", str(i + 1)]
                if not use_cuda:
                    cmd.append("--no-cuda")
                procs.append(subprocess.Popen(cmd, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL))
            a = Arguments()
            a.model, a.batch_size, a.epochs, a.lr, a.loss = model, bsz, epochs, args.lr, "bce"
            clock = FakeClock()
            c = Coordinator(1, True, rounds, False, False, args=a, transport="tcp", timer_factory=clock,
                            path=os.path.join(tmp, "test.pth"), device=torch.device("cuda", 0) if use_cuda else torch.device("cpu"))
            c.connect("127.0.0.1", broker.port)
            c.subscribe(topic)
            c.loop_start()
            pub = BusClient("bench-devices", transport="tcp")
            pub.connect("127.0.0.1", broker.port)
            pub.loop_start()
            deadline = time.time() + 120                 # first `import torch` of the worker processes can take a while
            from colearn_federated_learning_b200 import settings
            while len(settings.training_devices) < n_workers and time.time() < deadline:
                time.sleep(0.05)
            assert len(settings.training_devices) == n_workers, "the worker processes did not announce themselves"

            def one_training() -> float:
                t0 = time.perf_counter()
                clock.advance(1.0)                        # the window closes: select, 12 rounds over TCP, FedAvg, save
                dt = time.perf_counter() - t0
                res = c.windower.last_result
                assert res is not None and res["rounds"] == rounds and not res["dropped"], res
                for port in ports:                        # the devices ask again (mosquitto_pub in the reference's README)
                    pub.publish(topic, f"(127.0.0.1, {port}, TRAINING)")
                t_end = time.time() + 10
                while len(settings.training_devices) < n_workers and time.time() < t_end:
                    time.sleep(0.002)
                return dt

            for _ in range(W):
                one_training()
            times = [one_training() for _ in range(K)]
            final_losses = dict(c.windower.last_result["losses"])
            c.loop_stop()
            pub.loop_stop()
        finally:
            for p in procs:
                p.terminate()
            for p in procs:
                try:
                    p.wait(timeout=10)
                except subprocess.TimeoutExpired:
                    p.kill()
            broker.stop()
    total_s = sum(times)
    if full:      # one round = one full epoch of batch-1 SGD on the worker: the paper's figure of merit is steps/s
        steps_s = per_worker * K / total_s
        print(json.dumps({
            "metric": "batch-1 SGD steps/sec through the remote-mode stack (1 worker process, full epoch, host clock)",
            "value": steps_s, "unit": "steps/s", "n_gpus": 1 if use_cuda else 0, "steps": K, "warmup": W, "ms_per_step": total_s / K * 1e3,
            "higher_is_better": True, "scaling": "n/a", "vs_baseline": steps_s / 163.7, "dtype": "fp32",
            "data": "synthetic UNSW-IoT-shaped features / random-init weights", "impl": "ours",
            "config": {"name": "fulldata", "model": model, "description": desc, "samples": per_worker, "batch_size": bsz, "rounds": 1,
                       "total_training_time_s": total_s / K, "published_total_training_time_s": 4481.6,
                       "worker_device": "cuda (persistent kernel)" if use_cuda else "cpu (native host executor)",
                       "baseline_ref": "163.7 SGD steps/s: 733 672 samples in 4 481.6 s on 1x RPi 3B+ (BASELINE.md)"},
            "e2e": {"value": steps_s, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                    "timing": "the measurement is already end to end (host clock around whole trainings incl. the TCP round trip)"},
            "gpu_launches": K if use_cuda else 0}))
        return
    value = rounds * K / total_s
    print(json.dumps({
        "metric": "FL rounds/sec (remote mode, 2 worker processes over TCP, 1000 batch-1 iterations per round, host clock)",
        "value": value, "unit": "rounds/s", "n_gpus": 1 if use_cuda else 0, "steps": K, "warmup": W,
        "ms_per_step": total_s / K * 1e3, "higher_is_better": True, "scaling": "n/a", "vs_baseline": value / PUBLISHED_ROUNDS_PER_S,
        "dtype": "fp32", "data": "synthetic UNSW-IoT-shaped features / random-init weights", "impl": "ours",
        "config": {"name": "paper", "model": model, "description": desc, "rounds_per_training": rounds, "workers": n_workers,
                   "local_iterations_per_round": 1000, "samples_per_worker": per_worker, "loss": "bce", "batch_size": bsz,
                   "total_training_time_s": total_s / K, "published_total_training_time_s": 105.921,
                   "seconds_per_round": total_s / K / rounds, "published_seconds_per_round": 8.827,
                   "worker_device": "cuda (persistent kernel)" if use_cuda else "cpu (native host executor)",
                   "final_losses": {k: float(v) for k, v in final_losses.items()},
                   "bytes_coordinator_to_workers_per_round": c.windower.last_result.get("bytes_out", 0) // rounds,
                   "bytes_workers_to_coordinator_per_round": c.windower.last_result.get("bytes_in", 0) // rounds,
                   "published_bytes_per_round": "~72 kB to 2 workers, ~30.6 kB back per worker (paper §4.3)",
                   "baseline_ref": "0.1133 rounds/s = 12 rounds x 1000 it on 2x RPi 3B+ (BASELINE.md)"},
        "e2e": {"value": value, "unit": "rounds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "timing": "the measurement is already end to end (host clock around whole trainings, model shipped over TCP both ways every round)"},
        "gpu_launches": (2 * rounds * K) if use_cuda else 0}))


def bench_smpc(args) -> None:
    """Encrypted training (fixed-point additive sharing, Beaver triples, shared ReLU / cubic sigmoid) of the reference
    FFNN on ``n_train_items`` samples, batch 1 — what ``federated_coordinator.py -e`` runs after its window closes.  The
    paper only gives a figure for this (Fig. 7: up to ~600 s for 1000 items with SPDZ + SecureNN on a MacBook)."""
    import contextlib
    import io

    import torch

    from colearn_federated_learning_b200.control.arguments import Arguments
    from colearn_federated_learning_b200.data import BaseDataset, synthetic_unsw
    from colearn_federated_learning_b200.fl.encrypted import train_encrypted
    from colearn_federated_learning_b200.models import build_model

    model, items, bsz, epochs, _, desc = CONFIGS["smpc"]
    items = args.samples or items
    K, W = max(1, args.steps), max(1, min(args.warmup, 3))
    a = Arguments()
    a.n_train_items_enc, a.batch_size, a.epochs, a.lr = items, args.batch_size or bsz, args.local_epochs or epochs, args.lr
    x, y = synthetic_unsw(2 * items, seed=0)
    ds = BaseDataset(x, y)
    times, info = [], {}
    for i in range(W + K):
        torch.manual_seed(1)
        m = build_model(model)
        with contextlib.redirect_stdout(io.StringIO()):
            t0 = time.perf_counter()
            info = train_encrypted(m, ds, ["192.168.1.7", "192.168.1.8"], a)
            dt = time.perf_counter() - t0
        if i >= W:
            times.append(dt)
    per_training = sum(times) / len(times)
    value = items / per_training
    print(json.dumps({
        "metric": "SMPC-encrypted training throughput (secret-shared samples/s, 2 workers + crypto provider, host clock)",
        "value": value, "unit": "samples/s", "n_gpus": 0, "steps": K, "warmup": W, "ms_per_step": per_training * 1e3,
        "higher_is_better": True, "scaling": "n/a", "vs_baseline": value / (1000.0 / 600.0), "dtype": "int64 fixed point (3 fractional digits)",
        "data": "synthetic UNSW-IoT-shaped features / random-init weights", "impl": "ours",
        "config": {"name": "smpc", "model": model, "description": desc, "items": items, "batch_size": a.batch_size,
                   "seconds_per_training": per_training, "beaver_triples": info.get("triples"), "comparisons": info.get("comparisons"),
                   "baseline_ref": "paper Fig. 7 (figure only): up to ~600 s for 1000 items, MacBook, PySyft SPDZ + SecureNN"},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "timing": "host clock around whole encrypted trainings (sharing of data and model included)"},
        "gpu_launches": 0}))


def load_ref_local_data(total: int, rank: int, world: int):
    """The config both bench arms share: the synthetic Bot-IoT CSV the reference arm trains on (written by the same
    numpy-only generator, same seed), read through THIS repo's ``NetworkTrafficDataset`` (CSV -> feature selection -> MinMax),
    split into ``world`` contiguous shards like ``dataset.federate(workers)`` (fc.py:347-350)."""
    import tempfile

    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    from reference_arm import write_synthetic_csv
    from colearn_federated_learning_b200.data import NetworkTrafficDataset, shard_bounds

    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "synthetic_unsw.csv")
        write_synthetic_csv(path, total, seed=0)
        x, y = NetworkTrafficDataset(path).tensors()
    lo, hi = shard_bounds(total, world)[rank]
    return x[lo:hi].contiguous(), y[lo:hi].contiguous()


def run_engine_config(args, name: str, rank: int, world: int, device, full: bool = True):
    """Measure one GPU config through ``FederatedEngine``; returns the JSON record on rank 0 (None elsewhere).
    ``full=False``: the short form attached to the default line for a second config (no e2e-sync / self-check extras)."""
    import torch
    import torch.distributed as dist
    from colearn_federated_learning_b200 import ops
    from colearn_federated_learning_b200.parallel import FederatedEngine
    from colearn_federated_learning_b200.utils.monitors import NvmlSampler

    model, total, bsz, epochs, select_k, desc = CONFIGS[name]
    total = args.samples or total
    bsz = args.batch_size or bsz
    epochs = args.local_epochs or epochs
    K, W = args.steps, max(3, args.warmup)
    ref_local = name == "ref_local"
    x, y = load_ref_local_data(total, rank, world) if ref_local else make_data(model, total, rank, world)
    n_local = x.shape[0]
    mask = None
    if select_k is not None and select_k < world:
        mask = (1 << select_k) - 1  # registration order = rank order ("first" policy)
    flush_buf = None if args.no_flush else torch.empty(160 * 1024 * 1024 // 4, device=device)  # 160 MB > 126 MB L2

    def max_over_ranks(v: float) -> float:
        t = torch.tensor([v], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # reference local mode: sum-squared-error (cf.py:112), uniform FedAvg (PySyft federated_avg); BASELINE configs: n_k weights
    engine = FederatedEngine(model, backend="fused", device=device, batch_size=bsz, lr=args.lr, local_epochs=epochs,
                             weighted=not ref_local, loss="sse" if ref_local else "auto", seed=1, bf16_shadow=(model == "wide_mlp"))
    engine.set_local_data(x, y)
    for _ in range(W):
        engine.run_rounds(1, masks=mask)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = NvmlSampler(index=device.index or 0, period_s=0.02)
    sampler.start()
    dev_ms, launches = 0.0, 0
    for _ in range(K):
        if flush_buf is not None:
            ops.l2_flush(flush_buf)
        rep = engine.run_rounds(1, masks=mask)
        dev_ms += rep.device_ms
        launches += rep.launches
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop()
    # what the last timed round gave its caller, kept before the untimed passes below move the model on
    last_outputs = {"theta": engine.global_flat().clone(), "losses": rep.losses}
    dev_ms = max_over_ranks(dev_ms)
    extra = dict(rep.extra)
    # K rounds enqueued in one call: no host in the loop, no flush (what a training of K rounds costs on the device)
    rep_p = engine.run_rounds(K, masks=mask)
    extra["pipelined_rounds_per_s"] = K / (max_over_ranks(rep_p.device_ms) * 1e-3)
    extra["final_mean_loss"] = float(rep_p.losses[-1, :, 1].mean()) if (rep_p.losses is not None and rank == 0) else None

    e2e = None
    if not args.no_e2e:
        hx, hy = x.pin_memory(), y.pin_memory()
        h2d = int(hx.numel() * hx.element_size() + hy.numel() * hy.element_size())
        d2h = int(engine.loss_host.numel() * 4) if rank == 0 else 8

        def timed(fn) -> float:
            fn(2)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            fn(K)
            torch.cuda.synchronize()
            return max_over_ranks(time.perf_counter() - t0)

        def per_call(k):       # one public-API call per round: H2D of the round's shard, the round, D2H of its losses, host sync
            for _ in range(k):
                engine.run_rounds(1, masks=mask, host_inputs=[(hx, hy)], read_back=True, barrier=False)

        def one_call(k):       # the same k rounds in ONE call: every round still copies its inputs in and its losses out, the host
            engine.run_rounds(k, masks=mask, host_inputs=[(hx, hy)] * k, read_back="pipelined", barrier=False)   # reads them one round late

        wall_sync = timed(per_call)
        if engine.algo == "star":
            wall = timed(one_call)
            losses_read = len(engine.loss_history) if rank == 0 else None
            e2e = {"value": K / wall, "unit": "rounds/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                   "timing": "host clock around ONE run_rounds(K) call, max over ranks, sync both sides; every round copies its shard "
                             "H2D from pinned memory and its losses D2H; the host reads round i's losses while round i+1 runs",
                   "losses_read_on_host": losses_read, "per_call_sync_value": K / wall_sync}
        else:
            e2e = {"value": K / wall_sync, "unit": "rounds/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                   "timing": "host clock, one run_rounds(1) call per round with a host sync after its D2H, max over ranks"}

    check = None
    if full:
        check = engine.verify_round(mask)        # fused round vs dist.broadcast + same local fit + dist.reduce, same inputs
    nvlink = None
    if full and getattr(args, "nvlink_counters", False) and world > 1:
        import time as _time
        from colearn_federated_learning_b200.utils.monitors import NvlinkCounters
        ctr = NvlinkCounters(index=device.index or 0, uuid=str(torch.cuda.get_device_properties(device).uuid))
        if ctr.ok:
            dist.barrier()
            torch.cuda.synchronize()
            _time.sleep(0.3)
            a = ctr.read()
            engine.run_rounds(K, masks=mask)
            torch.cuda.synchronize()
            dist.barrier()
            torch.cuda.synchronize()
            _time.sleep(0.3)
            d = ctr.delta(a, ctr.read())
            mine = torch.tensor([d["tx_bytes"] / K, d["rx_bytes"] / K] if d else [-1.0, -1.0], device=device, dtype=torch.float64)
            allr = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(allr, mine)
            nvlink = {"counter": "NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX/RX over all links of each rank's GPU (payload bytes), untimed extra pass of K rounds",
                      "tx_bytes_per_round_by_rank": [float(t[0]) for t in allr], "rx_bytes_per_round_by_rank": [float(t[1]) for t in allr],
                      "model_bytes": int(engine.P) * 4, "algo": engine.algo}
        else:
            nvlink = {"unavailable": ctr.err}

    value = K / (dev_ms * 1e-3)
    if rank != 0:
        return None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, name, last_outputs)
    steps_per_round = epochs * ((n_local + bsz - 1) // bsz)
    cfg = {"name": name, "model": model, "description": desc, "global_batch": bsz * world,
           "batch_size_per_worker": bsz, "seq_len": None, "parallelism": f"fedavg-dp{world}",
           "total_samples": total, "samples_per_worker": n_local, "local_epochs": epochs,
           "local_sgd_steps_per_round": steps_per_round, "selected_workers": select_k or world,
           "loss": engine.cfg.loss, "lr": args.lr,
           "fedavg": "uniform (reference federated_avg)" if ref_local else "sample-count weighted",
           "l2": "flushed between timed rounds (160 MB write)" if flush_buf is not None else "not flushed",
           "shuffle": "keyed Feistel order computed inside the worker kernel every round (inside the timed region)",
           "baseline_ref": "0.1133 rounds/s = 12 rounds x 1000 it on 2x RPi 3B+ (BASELINE.md)",
           "switches": {k: v for k, v in sorted(os.environ.items()) if k.startswith("COLEARN_")}, **extra}
    if check is not None:
        cfg["self_check"] = check
    if nvlink is not None:
        cfg["nvlink"] = nvlink
    if engine.algo == "twoshot":
        # roofline of the round (BASELINE.json: "the slower of its compute at peak and its bytes over NVLink at link bandwidth"):
        # compute = the rank's local fit (MLP: 6 FLOP per parameter and sample) at the MEASURED bf16 matmul peak; link = the
        # all-reduce-with-broadcast of the arena through one GPU's NVLink port, (W-1)/W of the model per direction, fp32 in and
        # fp32 + bf16 shadow out, at 900 GB/s per direction
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except OSError:
            pass
        peak_tflops = float(peaks.get("bf16_tflops", 1693.2))
        P = engine.P
        flops = 6.0 * P * n_local * epochs if model == "wide_mlp" else None
        out_bytes = P * (4 + (2 if engine.bf16_shadow else 0))
        link_bytes = (world - 1) / world * max(P * 4, out_bytes)
        t_compute = flops / (peak_tflops * 1e12) * 1e3 if flops else None
        t_link = link_bytes / 900e9 * 1e3
        bound = max(t_compute or 0.0, t_link)
        ms = dev_ms / K
        cfg["roofline"] = {"compute_ms_at_measured_peak": t_compute, "peak_bf16_tflops": peak_tflops, "link_ms_at_900GBps_per_dir": t_link,
                           "link_bytes_per_dir_per_gpu": int(link_bytes), "bound_ms": bound, "roofline_frac": (bound / ms) if bound else None,
                           "achieved_tflops_per_gpu": (flops / (ms * 1e-3) / 1e12) if flops else None,
                           "note": "frac = max(compute at peak, bytes at link rate) / measured round time"}
    return {
        "metric": "FL rounds/sec (whole box, device-timed, max over ranks)",
        "value": value, "unit": "rounds/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": value / PUBLISHED_ROUNDS_PER_S,
        "dtype": "bf16" if model in ("resnet18", "wide_mlp") else "fp32",
        "data": ("synthetic UNSW-IoT-shaped CSV (Bot-IoT 10-best header) / random-init weights" if ref_local else
                 "synthetic UNSW-IoT-shaped features / random-init weights" if model != "resnet18"
                 else "synthetic 32x32 images / random-init weights"),
        "impl": "ours", "config": cfg,
        "clocks": {"sm_mhz": clocks.get("sm_mhz"), "sm_max_mhz": clocks.get("sm_max_mhz"), "reasons": clocks.get("reasons", []),
                   "power_w_max": clocks.get("power_w_max"), "samples": clocks.get("samples")},
        "e2e": e2e, "gpu_launches": launches,
    }


def run_torch_nccl(args, name: str, rank: int, world: int, device):
    """The stock-PyTorch + NCCL comparator (baseline/torch_nccl_fedavg.py) on the same config."""
    import torch
    import torch.distributed as dist
    from baseline.torch_nccl_fedavg import TorchNcclFedAvg
    from colearn_federated_learning_b200.models import build_model, DEFAULT_LOSS
    from colearn_federated_learning_b200.utils.monitors import NvmlSampler

    model, total, bsz, epochs, select_k, desc = CONFIGS[name]
    total, bsz, epochs = args.samples or total, args.batch_size or bsz, args.local_epochs or epochs
    K, W = args.steps, max(3, args.warmup)
    ref_local = name == "ref_local"
    x, y = load_ref_local_data(total, rank, world) if ref_local else make_data(model, total, rank, world)
    mask = (1 << select_k) - 1 if (select_k is not None and select_k < world) else None
    flush_buf = None if args.no_flush else torch.empty(160 * 1024 * 1024 // 4, device=device)

    def max_over_ranks(v: float) -> float:
        t = torch.tensor([v], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    torch.manual_seed(1)
    eng = TorchNcclFedAvg(build_model(model), device, loss="sse" if ref_local else DEFAULT_LOSS[model], batch_size=bsz, lr=args.lr,
                          epochs=epochs, weighted=not ref_local, bf16_autocast=(model in ("resnet18", "wide_mlp")))
    eng.set_local_data(x, y)
    hx, hy = x.pin_memory(), y.pin_memory()
    for _ in range(W):
        eng.run_round(mask)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = NvmlSampler(index=device.index or 0, period_s=0.02)
    sampler.start()
    dev_ms = 0.0
    for _ in range(K):
        if flush_buf is not None:
            flush_buf.fill_(1.0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        eng.run_round(mask)
        e1.record()
        torch.cuda.synchronize()
        dev_ms += e0.elapsed_time(e1)
    if world > 1:
        dist.barrier()
    clocks = sampler.stop()
    dev_ms = max_over_ranks(dev_ms)
    e2e = None
    if not args.no_e2e:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(K):
            eng.run_round(mask, host_inputs=(hx, hy))
        torch.cuda.synchronize()
        wall = max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": K / wall, "unit": "rounds/s",
               "h2d_bytes_per_step": int(hx.numel() * hx.element_size() + hy.numel() * hy.element_size()),
               "d2h_bytes_per_step": 4, "timing": "host clock, max over ranks, sync both sides"}
    if rank != 0:
        return None
    value = K / (dev_ms * 1e-3)
    return {"metric": "FL rounds/sec (whole box, device-timed, max over ranks)", "value": value, "unit": "rounds/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": value / PUBLISHED_ROUNDS_PER_S, "dtype": "bf16" if model in ("resnet18", "wide_mlp") else "fp32",
            "data": "synthetic / random-init weights", "impl": "torch_nccl_comparator",
            "config": {"name": name, "model": model, "description": desc, "total_samples": total, "samples_per_worker": int(x.shape[0]),
                       "batch_size_per_worker": bsz, "local_epochs": epochs, "parallelism": f"fedavg-dp{world}",
                       "l2": "flushed between timed rounds" if flush_buf is not None else "not flushed",
                       "shuffle": "torch.randperm on the host + H2D every round (inside the timed region)"},
            "clocks": {"sm_mhz": clocks.get("sm_mhz"), "sm_max_mhz": clocks.get("sm_max_mhz"), "reasons": clocks.get("reasons", [])},
            "e2e": e2e, "gpu_launches": 0}


def main() -> None:
    args = parse_args()
    if args.impl == "reference":
        # the unmodified reference from oracle/_ref on its own stock path; nothing of this repo's package is imported
        sys.path.insert(0, os.path.join(ROOT, "baseline"))
        import reference_arm
        reference_arm.main(args)
        return
    default_line = args.config is None
    name = args.config or "ref_local"
    if name == "cfg1":
        bench_cfg1(args)
        return
    if name in ("paper", "fulldata"):
        args.config = name
        bench_paper(args)
        return
    if name == "smpc":
        bench_smpc(args)
        return

    from colearn_federated_learning_b200.parallel import init_distributed, shutdown

    rank, world, device = init_distributed()
    if world != args.gpus and rank == 0:
        print(f"[bench] warning: --gpus {args.gpus} but WORLD_SIZE={world}; using {world}", file=sys.stderr)
    if device.type != "cuda":
        print(json.dumps({"impl": args.impl, "unavailable": "no CUDA device on this box"}))
        return
    if args.impl == "torch_nccl":
        out = run_torch_nccl(args, name, rank, world, device)
    else:
        out = run_engine_config(args, name, rank, world, device)
        if default_line:
            # the default line is the config BOTH arms can run (the reference's own model and local-training path); BASELINE.json's
            # config 2 (MLP 10-64-64-2, n_k-weighted) is measured in the same process and attached, so the round-1 headline
            # (BENCH_r01: cfg2) stays comparable
            also = run_engine_config(args, "cfg2", rank, world, device, full=False)
            if out is not None and also is not None:
                out["config"]["also_measured"] = {"cfg2": {k: also[k] for k in ("value", "unit", "ms_per_step", "e2e", "gpu_launches")}
                                                  | {"description": also["config"]["description"],
                                                     "pipelined_rounds_per_s": also["config"].get("pipelined_rounds_per_s")}}
    if rank == 0 and out is not None:
        print(json.dumps(out))
    shutdown()


def _keep_stdout_for_the_result_line() -> None:
    """The contract is ONE JSON line on stdout.  Libraries write to file descriptor 1 behind Python's back (NCCL prints its
    version banner there at world > 1), so fd 1 is pointed at stderr for the life of the process and Python's ``sys.stdout``
    — what ``print`` of the result line uses — keeps the original stream."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real, "w", buffering=1)


if __name__ == "__main__":
    _keep_stdout_for_the_result_line()
    main()

"""Per-SGD-step cost of the generic persistent MLP kernel (ops/csrc/mlp_generic.cu) against the layer-wise tcgen05 trainer.

    python scripts/bench_generic_mlp.py --out DIR [--n 8192] [--reps 10]

Measures, with CUDA events (warm-up, then the median of --reps launches) on --n samples (8192, as bench.py's ref_local config):
  * Net 784-128-64-10 (xent) and a plugin-shaped 10-96-48-1 (sigmoid, bce) at batch 1, 2, 4, 8, 16, 32: the generic kernel at
    every legal cluster size and LayerwiseMLPTrainer in the same config, alternated in this process;
  * the FFNN dims (10-50-30-10-1) through the generic kernel next to the specialised v6 kernel (the cost of generality);
  * a 37-client VirtualWorker launch of Net (37 x C CTAs).
The layer-wise trainer runs a capped number of steps (--lw-steps) per timed fit: its per-step cost does not depend on the
position in the epoch, and a full 8192-step batch-1 fit takes seconds.  Prints the card name and power limit and writes
DIR/generic_mlp.json.  Needs a GPU: there is no CPU fallback.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from colearn_federated_learning_b200 import ops  # noqa: E402
from colearn_federated_learning_b200.fl.layerwise import LayerwiseMLPTrainer  # noqa: E402
from colearn_federated_learning_b200.fl.trainer import FitConfig  # noqa: E402
from colearn_federated_learning_b200.models.mlp import MLPSpec  # noqa: E402
from colearn_federated_learning_b200.ops import reference  # noqa: E402

MODELS = {"net": ((784, 128, 64, 10), "none", "xent"), "plugin": ((10, 96, 48, 1), "sigmoid", "bce")}
FFNN = ((10, 50, 30, 10, 1), "sigmoid", "bce")
BATCHES = (1, 2, 4, 8, 16, 32)


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    parts = [p.strip() for p in line.split(",")] if line else []
    return {"name": parts[0] if parts else torch.cuda.get_device_name(0), "power_limit": parts[1] if len(parts) > 1 else "unknown",
            "max_sm_clock": parts[2] if len(parts) > 2 else "unknown"}


def data(dims, loss, n, dev, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(n, dims[0], generator=g)
    y = (torch.randint(0, dims[-1], (n, 1), generator=g).float() if loss == "xent"
         else (torch.rand(n, dims[-1], generator=g) > 0.5).float())
    return x.to(dev).contiguous(), y.to(dev).contiguous()


def timed(fn, reps: int, warmup: int) -> float:
    """Median milliseconds of fn() over reps launches (CUDA events around each)."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return statistics.median(times)


def generic_launcher(dims, act, loss, x, y, theta, batch, cluster, n_clients=1, specialised=False):
    dev = x.device
    slots = theta.unsqueeze(0).repeat(n_clients, 1).contiguous()
    loss_out = torch.zeros(n_clients, 2, device=dev)
    tasks = [ops.ClientTask(x=x, y=y, theta_in=theta, theta_out=slots[i], loss_out=loss_out[i]) for i in range(n_clients)]
    descs = ops.build_client_descs(tasks, dev)
    ext = ops._ext.require()
    if specialised:
        kind = ops.net_kind_for(dims, act)
        return lambda: ext.mlp_local_sgd(kind, descs, 0, n_clients, batch, 1, -1, ops.LOSS_CODES[loss], 0.01,
                                         ops.fused_mlp.resolve_variant(kind))
    return lambda: ext.mlp_local_sgd_generic(list(dims), act == "sigmoid", descs, 0, n_clients, batch, 1, -1, ops.LOSS_CODES[loss],
                                             0.01, cluster)


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--n", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--lw-steps", type=int, default=256)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_generic_mlp needs a GPU")
    dev = torch.device("cuda", 0)
    info = card()
    print(f"card: {info['name']}, power limit {info['power_limit']}, max SM clock {info['max_sm_clock']}", flush=True)
    res = {"card": info, "n": args.n, "reps": args.reps, "lw_steps": args.lw_steps, "rows": []}

    for name, (dims, act, loss) in MODELS.items():
        x, y = data(dims, loss, args.n, dev)
        g = torch.Generator().manual_seed(1)
        P = sum(dims[i] * dims[i + 1] + dims[i + 1] for i in range(len(dims) - 1))
        theta = ((torch.rand(P, generator=g) * 2 - 1) * 0.05).to(dev)
        spec = MLPSpec(dims, act, loss)
        for b in BATCHES:
            steps = reference.total_steps(args.n, b, 1)
            clusters = [c for c in (1, 2, 4, 8) if ops.generic_plan(dims, act, b, c, loss) is not None]
            gens = {c: generic_launcher(dims, act, loss, x, y, theta, b, c) for c in clusters}
            lw_flat = theta.clone()
            tr = LayerwiseMLPTrainer(spec, lw_flat, b)
            lw_steps = min(steps, args.lw_steps)
            cfg = FitConfig(model=name, loss=loss, batch_size=b, lr=0.01, max_nr_batches=lw_steps, shuffle=False)

            def lw():
                tr.fit(lw_flat, x, y, cfg, None)
            row = {"model": name, "dims": list(dims), "batch": b, "steps": steps, "auto_cluster": ops.generic_plan(dims, act, b, 0, loss),
                   "generic_us_per_step": {}, "layerwise_us_per_step": []}
            # alternate the two in this process: generic at every C, then the layer-wise trainer, twice
            for _ in range(2):
                for c, fn in gens.items():
                    row["generic_us_per_step"].setdefault(str(c), []).append(1e3 * timed(fn, args.reps, args.warmup) / steps)
                row["layerwise_us_per_step"].append(1e3 * timed(lw, max(3, args.reps // 3), 1) / lw_steps)
            row["generic_us_per_step"] = {c: min(v) for c, v in row["generic_us_per_step"].items()}
            row["layerwise_us_per_step"] = min(row["layerwise_us_per_step"])
            best = min(row["generic_us_per_step"].items(), key=lambda kv: kv[1]) if row["generic_us_per_step"] else (None, None)
            row["best_cluster"], row["best_generic_us_per_step"] = best
            print(json.dumps(row), flush=True)
            res["rows"].append(row)

    # cost of generality: FFNN dims through the generic kernel vs the specialised v6 kernel
    dims, act, loss = FFNN
    x, y = data(dims, loss, args.n, dev, seed=3)
    P = sum(dims[i] * dims[i + 1] + dims[i + 1] for i in range(len(dims) - 1))
    theta = ((torch.rand(P, generator=torch.Generator().manual_seed(2)) * 2 - 1) * 0.1).to(dev)
    ffnn = {"specialised_us_per_step": 1e3 * timed(generic_launcher(dims, act, loss, x, y, theta, 1, 0, specialised=True),
                                                    args.reps, args.warmup) / args.n, "generic_us_per_step": {}}
    for c in (1, 2, 4, 8):
        if ops.generic_plan(dims, act, 1, c, loss) is not None:
            ffnn["generic_us_per_step"][str(c)] = 1e3 * timed(generic_launcher(dims, act, loss, x, y, theta, 1, c), args.reps,
                                                              args.warmup) / args.n
    print(json.dumps({"ffnn": ffnn}), flush=True)
    res["ffnn_cost_of_generality"] = ffnn

    # 37 VirtualWorkers of Net in one launch
    dims, act, loss = MODELS["net"]
    x, y = data(dims, loss, args.n // 8, dev, seed=4)
    P = sum(dims[i] * dims[i + 1] + dims[i + 1] for i in range(len(dims) - 1))
    theta = ((torch.rand(P, generator=torch.Generator().manual_seed(5)) * 2 - 1) * 0.05).to(dev)
    c = ops.generic_plan(dims, act, 1, 0, loss)
    one = 1e3 * timed(generic_launcher(dims, act, loss, x, y, theta, 1, c, n_clients=1), args.reps, args.warmup)
    many = 1e3 * timed(generic_launcher(dims, act, loss, x, y, theta, 1, c, n_clients=37), args.reps, args.warmup)
    vw = {"clients": 37, "cluster": c, "ctas": 37 * c, "samples_per_client": args.n // 8, "one_client_us": one, "launch_us": many,
          "us_per_step_per_client": many / (args.n // 8)}
    print(json.dumps({"virtual_workers": vw}), flush=True)
    res["virtual_workers_net"] = vw

    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "generic_mlp.json"), "w") as f:
        json.dump(res, f, indent=1)
    return 0


if __name__ == "__main__":
    sys.exit(main())

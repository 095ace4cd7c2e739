"""``federated_coordinator.py --box``: the reference's coordinator SERVICE mapped onto the GPUs of one box.

The reference coordinator subscribes, then serves forever (``federated_coordinator.py:294-300``): devices announce
``TRAINING`` / ``INFERENCE`` / ``NOT_READY``, the first ``TRAINING`` arms the temporal window (``:180-225``), the window
closes into a training over the snapshot of registered devices, the window re-arms (``:392,:597``), late joiners ride the
next window, ``NOT_READY`` withdraws a device (``:267-281``), ``INFERENCE`` runs the model on the device's tagged tensors
(``:227-265``).  Box mode keeps all of that and replaces the transport:

* every rank (= GPU) is a **device**: :class:`BoxAgent` publishes ``(10.0.0.<rank+1>, <8777+rank>, STATE)`` events;
* MQTT is replaced by the process group's key-value store (:class:`StoreRelay`, SURVEY K5): agents append events to a
  log in the store, a relay thread on rank 0 republishes them on the in-process bus, where the REAL control plane runs —
  event parser (+ allow-list), device registry, :class:`~..control.window.TemporalWindow`, selection policy
  (:class:`BoxControl`);
* what the coordinator decides travels back as **commands** in the same store (``train`` with the selection bitmask of
  the window that closed, ``inference`` for one rank, ``exit``); every rank's main thread executes them in order, because
  a training is collective: all ranks enter ``FederatedEngine.run_rounds`` where broadcast / local SGD / FedAvg are fused
  NVLink kernels (a rank that was not selected still serves the round's flags).

The loop ends after ``--exit-after N`` trainings (0 = until Ctrl-C), like the classic coordinator.
"""
from __future__ import annotations

import json
import logging
import os
import threading
import time
from typing import Any, Callable, Dict, List, Optional

import torch
import torch.distributed as dist

from ..control.arguments import Arguments, ROUND_MODE_BATCHES
from ..control.bus import BusClient, InProcessBroker
from ..control.event_parser import EventParser, format_event
from ..control.selection import SelectionPolicy, LOWER_BOUND, UPPER_BOUND
from ..control.window import TemporalWindow
from ..data import synthetic_for_model, NetworkTrafficDataset
from ..settings import DeviceRegistry
from ..utils.checkpoint import load_or_init, checkpoint_compatible
from ..models import flatten_params
from .engine import FederatedEngine
from .launcher import init_distributed, shutdown

log = logging.getLogger(__name__)

BASE_PORT = 8777
NVLINK_GBPS_PER_DIR = 900.0     # NVLink 5 per GPU and direction (the roofline the box-mode metrics refer to)


def rank_identity(rank: int):
    return f"10.0.0.{rank + 1}", BASE_PORT + rank


def worker_id_to_rank(worker_id: str) -> int:
    return int(worker_id.rsplit(":", 1)[1]) - BASE_PORT


# ---------------------------------------------------------------------------------------------------------------------
# transport: an append-only event log and an append-only command log in a key-value store
# ---------------------------------------------------------------------------------------------------------------------
class DictStore:
    """In-process stand-in for the c10d store (``set`` / ``get`` / ``add`` / ``check``): single-process box mode and tests."""

    def __init__(self) -> None:
        self._d: Dict[str, bytes] = {}
        self._n: Dict[str, int] = {}
        self._cv = threading.Condition()

    def set(self, key: str, value) -> None:
        with self._cv:
            self._d[key] = value if isinstance(value, bytes) else str(value).encode()
            self._cv.notify_all()

    def get(self, key: str) -> bytes:
        with self._cv:
            if not self._cv.wait_for(lambda: key in self._d, timeout=30):
                raise TimeoutError(key)
            return self._d[key]

    def add(self, key: str, amount: int) -> int:
        with self._cv:
            self._n[key] = self._n.get(key, 0) + int(amount)
            return self._n[key]

    def check(self, keys: List[str]) -> bool:
        with self._cv:
            return all(k in self._d for k in keys)


class StoreRelay:
    """Two logs on top of a store.  ``post(log, payload)``: ``seq = add(log/n, 1); set(log/seq, payload)``;
    ``poll(log)``: everything appended since this object last looked (in order).  One relay object per consumer."""

    def __init__(self, store, prefix: str = "colearn/box") -> None:
        self.store, self.prefix = store, prefix
        self._seen: Dict[str, int] = {}

    def post(self, logname: str, payload: str) -> int:
        seq = int(self.store.add(f"{self.prefix}/{logname}/n", 1))
        self.store.set(f"{self.prefix}/{logname}/{seq}", payload)
        return seq

    def poll_seq(self, logname: str) -> List[tuple]:
        """``[(seq, payload), ...]`` appended since this object last looked, in order."""
        n = int(self.store.add(f"{self.prefix}/{logname}/n", 0))
        out = []
        for seq in range(self._seen.get(logname, 0) + 1, n + 1):
            key = f"{self.prefix}/{logname}/{seq}"
            # the writer sets the entry right after taking its number.  A c10d store client holds its lock while a get
            # waits for a key, so when the writer is another thread of this process its set would wait for that get:
            # stop at the first entry not written yet and deliver it on a later poll
            if not self.store.check([key]):
                break
            v = self.store.get(key)
            out.append((seq, v.decode() if isinstance(v, (bytes, bytearray)) else str(v)))
            self._seen[logname] = seq
        return out

    def poll(self, logname: str) -> List[str]:
        return [p for _, p in self.poll_seq(logname)]

    def wait_next(self, logname: str, stop: Optional[Callable[[], bool]] = None, period_s: float = 0.002) -> Optional[tuple]:
        """Block until the log has an unread entry; returns ``(seq, payload)`` one at a time (None when ``stop()`` says so)."""
        buf = self.__dict__.setdefault("_buf", {}).setdefault(logname, [])
        while not buf:
            buf.extend(self.poll_seq(logname))
            if buf:
                break
            if stop is not None and stop():
                return None
            time.sleep(period_s)
        return buf.pop(0)


# ---------------------------------------------------------------------------------------------------------------------
# rank 0: the control plane
# ---------------------------------------------------------------------------------------------------------------------
class BoxControl:
    """Broker + parser + registry + temporal window + selection on rank 0.  ``pump()`` moves new device events from the
    store log onto the in-process bus (a thread calls it in :meth:`start`; tests call it by hand).  When a window closes,
    the selected devices become a ``train`` command; the window's timer thread then waits until rank 0's main thread has
    executed that command (``command_done``), so the window is in its TRAINING state for as long as the training runs and
    devices that announce meanwhile ride the next window — the reference's "keep" policy."""

    def __init__(self, relay: StoreRelay, world: int, window_s: float, topic: str, *, iot: bool = False,
                 select_k: Optional[int] = None, selection: str = "all", seed: int = 1, filter_file: Optional[str] = None,
                 strict: bool = False, timer_factory=None, rounds: int = 1, train_timeout_s: float = 3600.0) -> None:
        self.relay, self.world, self.topic, self.rounds = relay, world, topic, max(1, int(rounds))
        self.broker = InProcessBroker()
        self.registry = DeviceRegistry()
        kwargs = {"filter_file": filter_file} if filter_file else {}
        self.parser = EventParser(iot, strict=strict, **kwargs)
        self.policy = lambda: SelectionPolicy(LOWER_BOUND, UPPER_BOUND, selection, select_k, seed)
        self.windower = TemporalWindow(self.registry, window_s, self._window_closed, timer_factory, lower_bound=0,
                                       rearm_if_pending=True)
        self.train_timeout_s = train_timeout_s
        self.trainings_posted = 0
        self.inferences_posted = 0
        self.history: List[Dict[str, Any]] = []
        self._done: Dict[int, threading.Event] = {}
        self._cmd_lock = threading.Lock()
        self._stop = threading.Event()
        self._thread: Optional[threading.Thread] = None
        outer = self

        class _Sub(BusClient):
            def on_message(self, client, userdata, msg):
                outer._on_event(msg.payload)

        self.sub = _Sub("coordinator", broker=self.broker)
        self.sub.connect()
        self.sub.subscribe(topic)            # delivered by pump() (drain): one thread handles the events in log order
        self.pub = BusClient("store-relay", broker=self.broker)
        self.pub.connect()

    # -- device events ------------------------------------------------------------------------------------------------
    def _on_event(self, payload) -> None:
        ev = self.parser.parse(payload, remote=True)
        if ev is None:
            log.info("Event ignored: %r", payload)
            return
        rank = worker_id_to_rank(ev.worker_id)
        if not 0 <= rank < self.world:
            log.info("Event from an address that is not a rank of this box: %s", ev.worker_id)
            return
        if ev.state == "TRAINING":
            if self.windower.on_training(ev.worker_id, ev.worker_id):
                log.info("Timer starting")
        elif ev.state == "NOT_READY":
            log.info("%s is not ready anymore, removing from the known lists", ev.worker_id)
            self.windower.on_not_ready(ev.worker_id)
        elif ev.state == "INFERENCE":
            self.inferences_posted += 1
            self.post_command({"op": "inference", "rank": rank, "worker": ev.worker_id})
        log.info("ONMESSAGE: Training devices: %s", self.registry)

    def pump(self) -> int:
        """Republish the device events that arrived in the store since the last call; returns how many."""
        events = self.relay.poll("events")
        for payload in events:
            self.pub.publish(self.topic, payload)
        self.sub.drain()
        return len(events)

    def start(self, period_s: float = 0.005) -> None:
        def loop():
            while not self._stop.is_set():
                try:
                    self.pump()
                except Exception:  # noqa: BLE001 - the store goes away at shutdown
                    if self._stop.is_set():
                        return
                    log.exception("store relay failed")
                self._stop.wait(period_s)
        self._thread = threading.Thread(target=loop, name="box-store-relay", daemon=True)
        self._thread.start()

    def stop(self) -> None:
        self._stop.set()
        self.windower.cancel()
        if self._thread is not None:
            self._thread.join(timeout=2)

    # -- decisions -> commands ----------------------------------------------------------------------------------------
    def post_command(self, cmd: Dict[str, Any]) -> int:
        seq = self.relay.post("commands", json.dumps(cmd))
        return seq

    def _window_closed(self, snapshot) -> Optional[Dict[str, Any]]:
        sel = self.policy().select(snapshot)
        record = {"members": list(snapshot.keys()), "selected": list(sel.keys())}
        self.history.append(record)
        if not sel:
            log.info("No behaviour defined for the number of devices achieved")
            return None
        mask = 0
        for wid in sel:
            mask |= 1 << worker_id_to_rank(wid)
        log.info("window closed: members=%s selected=%s", record["members"], record["selected"])
        # the selected devices leave the registry now that their training starts (the reference removes them when it ends,
        # fc.py:573-580, and thereby loses a device that announced again meanwhile): a TRAINING event that arrives from here
        # on — a late joiner, or a trained device asking again — is a registration for the NEXT window
        for wid in sel:
            self.registry.remove(wid)
        self.trainings_posted += 1
        done = threading.Event()
        with self._cmd_lock:
            seq = self.post_command({"op": "train", "mask": mask, "rounds": self.rounds, "training": self.trainings_posted,
                                     "selected": record["selected"]})
            self._done[seq] = done
        if not done.wait(self.train_timeout_s):
            log.error("training %d did not finish within %.0f s", self.trainings_posted, self.train_timeout_s)
        with self._cmd_lock:
            self._done.pop(seq, None)
        record["mask"] = mask
        return record

    def command_done(self, seq: int) -> None:
        with self._cmd_lock:
            ev = self._done.get(seq)
        if ev is not None:
            ev.set()


# ---------------------------------------------------------------------------------------------------------------------
# every rank: the device
# ---------------------------------------------------------------------------------------------------------------------
class BoxAgent:
    """The device role of a rank: announces itself, optionally follows a script of further events.

    ``script`` items are ``(state, after_trainings)``: publish ``state`` once this rank has seen ``after_trainings``
    trainings complete (0 = right after the initial announcement) — how tests and ``--box-script`` inject NOT_READY,
    INFERENCE or late TRAINING events.  With ``reannounce`` the device asks for training again after every training it
    took part in (what a user does with ``mosquitto_pub`` in the reference's README)."""

    def __init__(self, relay: StoreRelay, rank: int, *, event: str = "TRAINING", reannounce: bool = True,
                 script: Optional[List[tuple]] = None) -> None:
        self.relay, self.rank, self.event, self.reannounce = relay, rank, event, reannounce
        self.script = sorted(script or [], key=lambda it: it[1])
        self.trainings_seen = 0

    def publish(self, state: str) -> None:
        ip, port = rank_identity(self.rank)
        self.relay.post("events", format_event(ip, state, port))

    def start(self) -> None:
        if self.event:
            self.publish(self.event)
        self._run_script()

    def _run_script(self) -> None:
        while self.script and self.script[0][1] <= self.trainings_seen:
            state, _ = self.script.pop(0)
            self.publish(state)

    def training_finished(self, took_part: bool, more_to_come: bool) -> None:
        self.trainings_seen += 1
        if took_part and self.reannounce and more_to_come:
            self.publish("TRAINING")
        self._run_script()


def parse_box_script(spec: Optional[str], rank: int) -> List[tuple]:
    """``"3:NOT_READY:0,2:INFERENCE:1"`` -> the ``(state, after_trainings)`` items of ``rank``."""
    out = []
    for item in (spec or "").split(","):
        item = item.strip()
        if not item:
            continue
        r, state, when = item.split(":")
        if int(r) == rank:
            out.append((state.strip().upper(), int(when)))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# the service
# ---------------------------------------------------------------------------------------------------------------------
def _c10d_store():
    from torch.distributed import distributed_c10d as c10d
    return c10d._get_default_store()


def round_record(round_idx: int, mask: int, world: int, counts: List[int], losses, device_ms: float, bytes_bcast: int,
                 bytes_reduce: int, launches: int, algo: str, phases: Optional[Dict[str, float]] = None) -> Dict[str, Any]:
    """One JSONL record per round (SURVEY §5 metrics): who trained, on how many samples, the losses, the device time
    (already the max over ranks), the per-phase device times of the coordinator rank when phase timing is on, the model
    bytes moved by the two collective legs and how far the round is from the time the slower leg would take at NVLink
    line rate."""
    sel = [k for k in range(world) if (mask >> k) & 1]
    t = max(device_ms, 1e-6) * 1e-3
    link_s = max(bytes_bcast, bytes_reduce) / (NVLINK_GBPS_PER_DIR * 1e9)
    rec = {"round": round_idx, "selected": ["%s:%d" % rank_identity(k) for k in sel], "n_k": [counts[k] for k in sel],
           "loss_k": [float(losses[k]) for k in sel], "t_round_max_over_ranks_ms": device_ms, "algo": algo,
           "bytes_bcast": bytes_bcast, "bytes_reduce": bytes_reduce, "launches": launches,
           "GBps": (bytes_bcast + bytes_reduce) / t / 1e9, "link_time_lower_bound_ms": link_s * 1e3,
           "roofline_frac": link_s / t}
    if phases:
        rec["phases_ms"] = phases
    return rec


def _run_rounds_observed(engine: FederatedEngine, mask: int, rounds: int, rank: int, world: int, metrics_path: Optional[str],
                         save_every: int, checkpoint: str, round0: int = 0) -> None:
    t0 = time.time()
    total_ms = 0.0
    for i in range(rounds):
        rep = engine.run_rounds(1, masks=mask)
        ms = torch.tensor([rep.device_ms], dtype=torch.float64, device=engine.device if engine.backend != "cpu" else "cpu")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        total_ms += float(ms)
        if rank == 0:
            losses = rep.losses[0, :, 0].tolist() if rep.losses is not None else [0.0] * world
            rec = round_record(round0 + i, mask, world, engine.counts, losses, float(ms), rep.bytes_bcast, rep.bytes_reduce,
                               rep.launches, rep.algo, rep.extra.get("phases_ms"))
            for k, l in zip([k for k in range(world) if (mask >> k) & 1], rec["loss_k"]):
                log.info("Loss for worker id: %s tensor(%.4f)", "%s:%d" % rank_identity(k), l)
            log.info("Time round %d : %s", i, rec["t_round_max_over_ranks_ms"] * 1e-3)
            if metrics_path:
                with open(metrics_path, "a") as f:
                    f.write(json.dumps(rec) + "\n")
            if save_every and (i + 1) % save_every == 0 and i + 1 < rounds:
                engine.save_checkpoint(checkpoint)
                log.info("checkpoint after round %d written to %s", i + 1, checkpoint)
    if rank == 0:
        log.info("Total training time: %s (device %.3f ms for %d rounds)", time.time() - t0, total_ms, rounds)


class BoxService:
    """What every rank runs after the process group is up: engine + device agent (+ control plane on rank 0) + the
    command loop."""

    def __init__(self, cli, args: Arguments, rank: int, world: int, device, store=None, timer_factory=None) -> None:
        self.cli, self.args, self.rank, self.world, self.device = cli, args, rank, world, device
        backend = args.backend
        if backend == "nccl":
            raise SystemExit("--box --backend nccl: the NCCL round is the comparator (bench.py --impl torch_nccl), not a box-mode "
                             "backend; use --backend fused (default on GPUs) or cpu")
        self.rounds = max(1, cli.federated_round)
        max_batches = args.federate_after_n_batches
        if self.rounds > 1 and max_batches < 0:
            max_batches = ROUND_MODE_BATCHES          # fc.py:533-535
        on_gpu = backend != "cpu" and device.type == "cuda"
        self.engine = FederatedEngine(args.model, backend=backend, device=device, batch_size=args.batch_size, lr=args.lr,
                                      local_epochs=args.epochs, max_batches=max_batches, loss=args.loss, weighted=args.weighted,
                                      server_lr=args.server_lr, seed=args.seed,
                                      bf16_shadow=on_gpu and getattr(args, "dtype", "fp32") == "bf16",
                                      clients_per_rank=getattr(cli, "clients_per_gpu", 1) if on_gpu else 1,
                                      round_deadline_ms=float(getattr(cli, "round_deadline_ms", 0.0) or 0.0))
        if rank == 0 and os.path.exists(cli.checkpoint) and checkpoint_compatible(self.engine.model, cli.checkpoint):
            load_or_init(self.engine.model, cli.checkpoint)
            self.engine.load_global(flatten_params(self.engine.model))
        # private shards: contiguous ceil(N/world) split of the dataset, like dataset.federate(workers)
        if args.synthetic and args.synthetic > 0:
            x, y = synthetic_for_model(args.model, args.synthetic, seed=args.seed)
        else:
            x, y = NetworkTrafficDataset(args.test_path).tensors()
        from ..data import shard_bounds
        lo, hi = shard_bounds(len(x), world)[rank]
        self.engine.set_local_data(x[lo:hi], y[lo:hi])
        self.eval_data = (x, y) if (rank == 0 and getattr(cli, "evaluate", False)) else None
        n_inf = int(getattr(cli, "box_inference_rows", 5) or 0)
        self.inference_x = x[lo:hi][:n_inf].clone()          # the device's "inference"-tagged tensors (rw.py:97-104)

        if store is None:
            store = _c10d_store() if (dist.is_available() and dist.is_initialized()) else DictStore()
        self.relay = StoreRelay(store)
        self.exit_after = int(getattr(cli, "exit_after", 0) or 0)
        self.agent = BoxAgent(StoreRelay(store), rank, event=getattr(cli, "box_event", "TRAINING") or "TRAINING",
                              reannounce=not getattr(cli, "box_no_reannounce", False),
                              script=parse_box_script(getattr(cli, "box_script", None), rank))
        self.control: Optional[BoxControl] = None
        if rank == 0:
            self.control = BoxControl(StoreRelay(store), world, float(cli.window), cli.topic, iot=cli.iot, select_k=cli.select,
                                      selection=cli.selection, seed=args.seed, filter_file=cli.filter_file, strict=cli.strict_events,
                                      timer_factory=timer_factory, rounds=self.rounds)
        self.trainings_done = 0
        self.rounds_done = 0
        self.last_predictions: Optional[List[int]] = None
        self.results: List[Dict[str, Any]] = []

    # -- commands -----------------------------------------------------------------------------------------------------
    def _train(self, cmd: Dict[str, Any]) -> None:
        mask, rounds = int(cmd["mask"]), int(cmd["rounds"])
        cli, rank, world = self.cli, self.rank, self.world
        t0 = time.time()
        save_every = max(0, getattr(self.args, "save_every", 0))
        metrics_path = getattr(cli, "metrics", None)
        if metrics_path or save_every:
            # observable mode: one engine call per round, so every round gets its own device time (max over ranks), traffic /
            # link-roofline figures and, if asked for, a checkpoint.  Without these flags all rounds are enqueued in one call
            _run_rounds_observed(self.engine, mask, rounds, rank, world, metrics_path, save_every, cli.checkpoint, self.rounds_done)
            losses = None
        else:
            rep = self.engine.run_rounds(rounds, masks=mask)
            losses = rep.losses
            if rank == 0:
                for i in range(rounds):
                    for k in range(world):
                        if (mask >> k) & 1:
                            log.info("Loss for worker id: %s tensor(%.4f)", "%s:%d" % rank_identity(k), float(rep.losses[i, k, 0]))
                log.info("Total training time: %s (device %.3f ms for %d rounds)", time.time() - t0, rep.device_ms, rounds)
        self.rounds_done += rounds
        self.trainings_done += 1
        result: Dict[str, Any] = {"training": self.trainings_done, "mask": mask, "rounds": rounds}
        if rank == 0:
            self.engine.save_checkpoint(cli.checkpoint)
            if losses is not None:
                result["final_losses"] = {("%s:%d" % rank_identity(k)): float(losses[-1, k, 0]) for k in range(world) if (mask >> k) & 1}
            if self.eval_data is not None:
                from ..fl.evaluate import evaluate
                x, y = self.eval_data
                ev = evaluate(self.engine.model, x.to(self.engine.device), y.to(self.engine.device),
                              flat=self.engine.global_flat().detach().clone(), verbose=False)
                result["eval_loss"] = ev["loss"]
                log.info("Loss evaluation global model after training: %s", ev["loss"])
        self.results.append(result)

    def _inference(self, cmd: Dict[str, Any]) -> None:
        """INFERENCE from rank ``r`` (fc.py:227-265): the global model goes to that device, the device runs it on its
        tagged tensors (``mlp_forward`` + ``argmax_rows`` on its GPU), the predictions come back to the coordinator."""
        r = int(cmd["rank"])
        theta = self.engine.global_flat().detach().clone()
        if self.world > 1:
            dist.broadcast(theta, src=self.engine.coord)
        box: List[Any] = [None]
        if self.rank == r:
            from ..fl.evaluate import predict
            box[0] = predict(self.engine.model, self.inference_x.to(theta.device), flat=theta).reshape(-1).tolist()
        if self.world > 1:
            dist.broadcast_object_list(box, src=r)
        self.last_predictions = box[0]
        if self.rank == 0:
            log.info("inference on %s: %s", cmd.get("worker"), box[0])

    # -- main loop ----------------------------------------------------------------------------------------------------
    def serve(self) -> List[Dict[str, Any]]:
        if self.control is not None:
            self.control.start()
        self.agent.start()
        try:
            while True:
                seq, raw = self.relay.wait_next("commands")
                cmd = json.loads(raw)
                if cmd["op"] == "exit":
                    break
                if cmd["op"] == "train":
                    self._train(cmd)
                    more = not (self.exit_after > 0 and self.trainings_done >= self.exit_after)
                    self.agent.training_finished(bool((int(cmd["mask"]) >> self.rank) & 1), more)
                    if self.control is not None:
                        if not more:
                            self.control.post_command({"op": "exit"})
                        self.control.command_done(seq)
                elif cmd["op"] == "inference":
                    self._inference(cmd)
        except KeyboardInterrupt:
            log.info("Coordinator stopped.")
        finally:
            if self.control is not None:
                self.control.stop()
        return self.results


def run_box_encrypted(cli, args: Arguments, rank: int, world: int, device) -> Optional[Dict[str, Any]]:
    """``--box -e``: the reference's encrypted demo (fc.py:394-472) with the roles on ranks — rank 0 = coordinator + crypto
    provider (dealer), two other ranks (ranks 1 and 2; ranks 0 and 1 on a 2-GPU box) = the share holders; one temporal window
    admits the devices, the first two share holders must be in it.  Shares travel dealer -> party point to point, the
    per-multiplication opens go party <-> party through this repo's P2P kernels on GPUs (``smpc/dist.py``)."""
    from ..models import MLPNet, build_model
    from ..smpc import PartyContext, train_encrypted_dist
    from ..utils.checkpoint import save_model

    store = _c10d_store() if (dist.is_available() and dist.is_initialized()) else DictStore()
    ctx = PartyContext(device, seed=args.seed)            # (collective: creates the pair's subgroup / exchange buffers)
    agent = BoxAgent(StoreRelay(store), rank, event=getattr(cli, "box_event", "TRAINING") or "TRAINING", reannounce=False)
    control = None
    if rank == 0:
        control = BoxControl(StoreRelay(store), world, float(cli.window), cli.topic, iot=cli.iot, selection="all", seed=args.seed,
                             filter_file=cli.filter_file, strict=cli.strict_events)
        control.start()
    agent.start()
    relay = StoreRelay(store)
    seq, raw = relay.wait_next("commands")
    cmd = json.loads(raw)
    result = None
    try:
        mask = int(cmd.get("mask", 0)) if cmd.get("op") == "train" else 0
        if not ((mask >> ctx.p0) & 1 and (mask >> ctx.p1) & 1):
            log.info("No behaviour defined for a number of workers less than 2 (share holders %d and %d must both be in the window)", ctx.p0, ctx.p1)
            return None
        torch.manual_seed(args.seed)
        model = build_model(args.model)
        if not isinstance(model, MLPNet):
            raise SystemExit("encrypted training supports the MLP family only")
        if rank == 0 and os.path.exists(cli.checkpoint) and checkpoint_compatible(model, cli.checkpoint):
            load_or_init(model, cli.checkpoint)
        n_items = int(args.n_train_items_enc)
        x = y = None
        if args.synthetic and args.synthetic > 0:
            xs, ys = synthetic_for_model(args.model, max(args.synthetic, n_items), seed=args.seed)
        else:
            xs, ys = NetworkTrafficDataset(args.test_path).tensors()
        n_items = min(n_items, len(xs))
        if ctx.is_dealer:
            order = torch.randperm(len(xs), generator=torch.Generator().manual_seed(args.seed))[:n_items]   # cf.py:269-277
            x, y = xs[order].to(device), ys[order].view(n_items, -1).to(device)
        if ctx.is_dealer or ctx.party is not None:
            model.to(device)
            log.info("Encryption and distribution of the model...")
            last, info = train_encrypted_dist(model, x, y, n_items, int(model.spec.dims[0]), int(model.spec.dims[-1]), args, ctx)
            if rank == 0:
                save_model(model.cpu(), cli.checkpoint, meta={"model": args.model, "mode": "encrypted-box", **{k: info[k] for k in ("dealer", "parties")}})
                log.info("End encryption: last loss %s, %d Beaver triples, %d comparisons, %.3f s", last, info["triples"], info["comparisons"], info["seconds"])
                result = {"last_loss": last, **info}
            elif ctx.party is not None:
                log.info("share holder %d: %d opens, %d bytes exchanged with the other share holder (%d through p2p_copy_kernel)",
                         ctx.party, info["opens"], info["bytes_between_parties"], info["p2p_opens"])
        return result
    finally:
        if control is not None:
            control.command_done(seq)
            control.stop()
        if dist.is_available() and dist.is_initialized():
            dist.barrier()


def run_box_coordinator(cli, args: Arguments) -> None:
    rank, world, device = init_distributed()
    try:
        if getattr(cli, "encryption", False):
            run_box_encrypted(cli, args, rank, world, device)
        else:
            BoxService(cli, args, rank, world, device).serve()
    finally:
        shutdown()

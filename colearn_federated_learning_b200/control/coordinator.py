"""The Coordinator: pub/sub subscriber + temporal-window scheduler + round loops.

Parity map (reference ``federated_coordinator.py``):
  ``Coordinator.__init__``  :93-124   bounds 1/2/100/2, ``./test.pth``, ``Arguments()``
  ``on_connect/on_publish`` :128-129, :291-292
  ``on_message``            :131-289  parse → worker handle → TRAINING / INFERENCE / NOT_READY
  ``run``                   :294-313  connect, subscribe qos 0, loop_forever, Ctrl-C cleanup
  ``starting_training_local`` :318-392, ``starting_training_enc`` :394-472,
  ``training_remote``       :475-597

Differences that are deliberate (SURVEY §2.8): the registry is locked; local mode is *true*
FedAvg (every worker starts the round from the same global θ) instead of averaging K aliases of
one module; INFERENCE uses the trained architecture; encrypted mode saves its model; Ctrl-C never
``KeyError``s; a failing/slow remote worker is dropped from the round instead of hanging it
(``fit_timeout``); selection at the upper bound is implemented, not just logged.
"""
from __future__ import annotations

import asyncio
import logging
import os
import time
from collections import OrderedDict
from typing import Any, Dict, List, Optional

import torch

from .. import ops, settings
from ..data import federate, synthetic_for_model, BaseDataset
from ..fl.fedavg import normalized_weights
from ..fl.trainer import FitConfig, local_fit, make_perm, resolve_loss
from ..fl.evaluate import evaluate
from ..models import MLPNet, build_model, flatten_params, unflatten_params
from ..utils.checkpoint import DEFAULT_PATH, checkpoint_compatible, load_or_init, save_model
from ..utils.metrics import RoundLogger
from .arguments import Arguments, ROUND_MODE_BATCHES
from .bus import BusClient, InProcessBroker, Message
from .event_parser import EventParser
from .selection import (LOWER_BOUND, LOWER_BOUND_ENC, UPPER_BOUND, UPPER_BOUND_ENC, SelectionPolicy)
from .window import TemporalWindow
from .workers import RemoteWorkerClient, VirtualWorker

log = logging.getLogger(__name__)


def default_device() -> torch.device:
    return torch.device("cuda" if torch.cuda.is_available() else "cpu")


class Coordinator(BusClient):
    def __init__(self, window: float, remote: bool, federated_round: int, encryption: bool,
                 iot_validation: bool, args: Optional[Arguments] = None, broker: Optional[InProcessBroker] = None,
                 transport: str = "inproc", timer_factory=None, path: str = DEFAULT_PATH,
                 strict_events: bool = False, device: Optional[torch.device] = None,
                 select_k: Optional[int] = None, selection: str = "all", fit_timeout: Optional[float] = None,
                 filter_file: Optional[str] = None, metrics: Optional[RoundLogger] = None,
                 rearm_if_pending: bool = False, evaluate_after: bool = False, worker_ssl_context=None) -> None:
        super().__init__(client_id="coordinator", broker=broker, transport=transport)
        self.worker_ssl_context = worker_ssl_context     # TLS towards the devices' RPC servers (control/tls.py)
        self.registry = settings.init()

        # Command parameters (fc.py:105-109)
        self.window = window
        self.remote = remote
        self.enabled_round = max(1, int(federated_round))
        self.encryption = encryption
        self.iot_validation = iot_validation

        # Other useful parameters (fc.py:112-124)
        kwargs = {"filter_file": filter_file} if filter_file else {}
        self.event_parser = EventParser(self.iot_validation, strict=strict_events, **kwargs)
        self.training_lower_bound = LOWER_BOUND
        self.training_lower_bound_enc = LOWER_BOUND_ENC
        self.training_upper_bound = UPPER_BOUND
        self.training_upper_bound_enc = UPPER_BOUND_ENC
        self.known_workers: Dict[str, Any] = {}   # the reference's ``server._known_workers``
        self.path = path
        self.args = args or Arguments()
        self.device = device or (torch.device("cpu") if self.args.no_cuda else default_device())
        self.select_k = select_k
        self.selection = selection
        self.fit_timeout = fit_timeout
        self.metrics = metrics or RoundLogger()
        self.evaluate_after = evaluate_after
        self.last_predictions: Optional[List[int]] = None
        self.trainings_done = 0
        self._in_flight: Dict[str, Any] = {}      # id -> handle of the devices a running training is using
        self._withdrawn: set = set()              # ids that sent NOT_READY while their fit was in flight

        self.windower = TemporalWindow(self.registry, window, self._start_training, timer_factory,
                                       lower_bound=0, rearm_if_pending=rearm_if_pending)

    # ------------------------------------------------------------------ paho-style callbacks
    def on_connect(self, mqttc, obj, flags, rc) -> None:
        log.info("Connected!")

    def on_publish(self, mqttc, obj, mid) -> None:
        log.info("mid: " + str(mid))

    def on_message(self, mqttc, obj, msg: Message) -> None:
        """One bus event (fc.py:131-289): decode it, build the device handle its state needs, run the state's handler
        from ``_STATE_HANDLERS``.  Malformed payloads, filtered addresses and unknown states end in one log line."""
        log.info("%s %s %s", msg.topic, msg.qos, msg.payload)
        event = self._decode_event(msg.payload)
        if event is None:
            log.info("Event ignored: payload is not a valid '(ip[, port], STATE)' tuple for this mode")
            return
        handler = self._STATE_HANDLERS[event["state"]]
        handle = None
        if event["state"] != "NOT_READY":
            handle = self._open_handle(event)
            if handle is None:
                return
        getattr(self, handler)(event, handle)
        log.info("ONMESSAGE: Training devices: " + str(self.registry))
        log.info("ONMESSAGE: All known workers: " + str(list(self.known_workers)))

    _STATE_HANDLERS = {"TRAINING": "_on_training", "INFERENCE": "_on_inference", "NOT_READY": "_on_not_ready"}

    def _decode_event(self, payload) -> Optional[Dict[str, Any]]:
        """``{ip, port, state, id}`` of a payload, or None.  Local events are ``(ip, STATE)``, remote ones
        ``(ip, port, STATE)``; the device id is ``ip`` / ``ip:port`` (fc.py:149,162)."""
        ev = self.event_parser.parse(payload, remote=self.remote)
        if ev is None:
            return None
        ident = f"{ev.ip}:{ev.port}" if self.remote else ev.ip
        return {"ip": ev.ip, "port": ev.port, "state": ev.state, "id": ident}

    def _open_handle(self, event: Dict[str, Any]):
        """The object a TRAINING / INFERENCE event registers: an in-process VirtualWorker, or a connection to the
        device's RPC server.  A device that cannot be reached is skipped (fc.py:166-170)."""
        if not self.remote:
            log.info("Local testing")
            return VirtualWorker(event["id"], self.device)
        log.info("Remote execution, worker id %s", event["id"])
        try:
            return RemoteWorkerClient(event["id"], event["ip"], event["port"], verbose=True, ssl_context=self.worker_ssl_context)
        except OSError as e:
            log.info("Device %s unreachable, skipped: %r", event["id"], e)
            return None

    def _on_training(self, event: Dict[str, Any], worker) -> None:
        # a device that announces twice (duplicate delivery, reconnect) replaces its handle; the old connection is closed
        # unless a training in flight is still using it (that one closes it itself)
        old = self.known_workers.get(worker.id)
        if old is not None and old is not worker and worker.id not in self._in_flight:
            self._close_quietly(old)
        self.known_workers[worker.id] = worker
        armed = self.windower.on_training(worker.id, worker)
        log.info(worker)
        if armed:
            log.info("Timer starting")

    def _on_inference(self, event: Dict[str, Any], worker) -> None:
        if self.remote:
            self._inference(worker)
        else:
            log.info("Inference is a remote-mode feature (local mode only tests the plumbing)")

    def _on_not_ready(self, event: Dict[str, Any], _worker) -> None:
        ident = event["id"]
        log.info("%s withdrew (NOT_READY): removing it from the known lists", ident)
        removed = self.windower.on_not_ready(ident)
        if removed is not None:
            if self._in_flight.get(ident) is removed:
                # its fit RPC is running and holds the connection's lock: closing here would block the bus thread until the
                # fit returns (forever for a hung device).  The training that uses the handle closes it when it finishes.
                self._withdrawn.add(ident)
                log.info("Worker %s is training right now; its connection is closed by that training", ident)
            else:
                self._close_quietly(removed)
        self.known_workers.pop(ident, None)

    @staticmethod
    def _close_quietly(handle) -> None:
        try:
            handle.close()
        except Exception:  # noqa: BLE001 - a dead socket must not take the bus thread down
            pass

    # ------------------------------------------------------------------ lifecycle
    def run(self, host: str, port: int, topic: str, forever: bool = True) -> None:
        self.connect(host, port)
        self.subscribe(topic, 0)
        log.info("Coordinator started. Press CTRL-C to stop")
        if not forever:
            self.loop_start()
            return
        try:
            self.loop_forever()
        except KeyboardInterrupt:
            self.shutdown()

    def shutdown(self) -> None:
        log.info("Coordinator stopped.")
        if self.windower.cancel():
            log.info("Cancelling the timer..")
        for key, worker in list(self.known_workers.items()):
            log.info("Closing socket for worker " + str(worker))
            try:
                worker.close()
            except Exception:  # noqa: BLE001
                pass
        self.loop_stop()
        log.info("Done")

    # ------------------------------------------------------------------ training dispatch
    def _start_training(self, snapshot: "OrderedDict[str, Any]") -> Any:
        from ..models.registry import num_params
        from ..utils.threads import small_model_threads
        self._in_flight = dict(snapshot)
        sizes = self.__dict__.setdefault("_param_counts", {})
        if self.args.model not in sizes:
            try:
                sizes[self.args.model] = num_params(build_model(self.args.model))
            except Exception:  # noqa: BLE001 - an unknown model fails later, with the proper message
                sizes[self.args.model] = 0
        try:
            # small models on the CPU: one intra-op thread (utils/threads.py: OpenMP fork/join costs more than the ops)
            with small_model_threads(sizes[self.args.model], self.device):
                return self._dispatch_training(snapshot)
        finally:
            self._in_flight = {}

    def _dispatch_training(self, snapshot: "OrderedDict[str, Any]") -> Any:
        if self.remote:
            loop = asyncio.new_event_loop()  # fresh loop inside the timer thread (fc.py:194-203)
            try:
                return loop.run_until_complete(self.training_remote(snapshot))
            finally:
                loop.close()
        if self.encryption:
            return self.starting_training_enc(snapshot)
        return self.starting_training_local(snapshot)

    def _policy(self, lower: int, upper: int, policy: Optional[str] = None) -> SelectionPolicy:
        return SelectionPolicy(lower_bound=lower, upper_bound=upper, policy=policy or self.selection,
                               select_k=self.select_k, seed=self.args.seed)

    def _load_model(self, name: Optional[str] = None):
        model = build_model(name or self.args.model)
        log.info("Loading model procedure started...")
        if os.path.exists(self.path) and not checkpoint_compatible(model, self.path):
            log.info("Checkpoint at %s does not match model %s; starting from a fresh model", self.path, name or self.args.model)
        else:
            load_or_init(model, self.path)
        log.info("Done")
        return model

    def _dataset(self):
        if self.args.synthetic and self.args.synthetic > 0:
            x, y = synthetic_for_model(self.args.model, self.args.synthetic, seed=self.args.seed)
            return BaseDataset(x, y)
        from ..data import load_dataset
        return load_dataset(getattr(self.args, "dataset", "unsw"), self.args.test_path)

    def _fit_config(self, mode: str) -> FitConfig:
        loss = self.args.loss
        if loss in ("auto", "", None):
            # reference: local mode trains with sum-squared-error (cf.py:112), remote with BCE (cf.py:79)
            loss = "sse" if (mode == "local" and self.args.model in ("ffnn", "testing_remote")) else resolve_loss(self.args.model, "auto")
        return FitConfig(model=self.args.model, loss=loss, batch_size=self.args.batch_size, epochs=self.args.epochs,
                         max_nr_batches=self.args.federate_after_n_batches, lr=self.args.lr, shuffle=True,
                         seed=self.args.seed)

    def _maybe_checkpoint(self, model, theta: torch.Tensor, round_idx: int, meta: Dict[str, Any]) -> None:
        """``--save-every N``: durable progress inside a long training (the reference only saves after the last
        round, fc.py:381,585).  Atomic like every checkpoint write; the final save still happens."""
        n = getattr(self.args, "save_every", 0)
        if n and (round_idx + 1) % n == 0 and round_idx + 1 < self.enabled_round:
            from ..models import state_dict_from_flat
            from ..utils.checkpoint import save_state_dict
            save_state_dict(state_dict_from_flat(model, theta), self.path, meta={**meta, "model": self.args.model, "rounds": round_idx + 1, "partial": True})
            log.info("checkpoint after round %d written to %s", round_idx + 1, self.path)

    def _deregister(self, trained) -> None:
        """Forget the devices that just trained (fc.py:376-379, 571-577) — unless the device re-announced itself
        while its training was running: that newer registration is a late joiner and rides the next window."""
        for wid in trained:
            used = self._in_flight.get(wid)
            current = self.registry.get(wid)
            if used is not None and current is not None and current is not used:
                log.info("Keeping " + str(wid) + ": it registered again during the training")
                continue
            log.info("Removing: " + str(wid) + " from training devices")
            self.registry.remove(wid)
            self.known_workers.pop(wid, None)

    # ------------------------------------------------------------------ local (VirtualWorker) mode
    def starting_training_local(self, snapshot: "OrderedDict[str, Any]") -> Optional[Dict[str, Any]]:
        to_train = self._policy(self.training_lower_bound, self.training_upper_bound).select(snapshot)
        if not to_train:
            log.info("No behaviour defined for the number of devices achieved")
            return None
        model = self._load_model()
        cfg = self._fit_config("local")

        log.info("Distribution data among the virtual workers")
        fed = federate(self._dataset(), list(to_train.keys()), self.device)
        log.info("Done")

        theta = flatten_params(model).to(self.device)
        model.to(self.device)
        log.info("Start training")
        self.metrics.start_training(cfg.max_nr_batches)
        result: Dict[str, Any] = {"workers": list(to_train.keys()), "losses": {}, "rounds": self.enabled_round}
        for r in range(self.enabled_round):
            t0 = time.time()
            flats, losses, counts = train_virtual_workers(theta, model, fed, cfg, r)
            live = [i for i, c in enumerate(counts) if c > 0]
            if live:
                w = normalized_weights([counts[i] for i in live] if self.args.weighted else None, len(live), device=self.device)
                ops.fedavg_apply(theta, flats[live].contiguous(), w, self.args.server_lr)
            for wid, l in zip(fed.workers, losses):
                self.metrics.worker_loss(wid, l)
                result["losses"][wid] = l
            self.metrics.end_round(r, time.time() - t0, selected=fed.workers, n_k=counts, loss_k=losses)
            self._maybe_checkpoint(model, theta, r, {"workers": fed.workers, "mode": "local"})
        log.info("End training")
        unflatten_params(model, theta)
        save_model(model.cpu(), self.path, meta={"model": self.args.model, "rounds": self.enabled_round, "workers": fed.workers, "mode": "local"})
        self._deregister(to_train.keys())
        self.metrics.end_training()
        self.trainings_done += 1
        log.info("End training local")
        return result

    # ------------------------------------------------------------------ encrypted (SMPC) mode
    def starting_training_enc(self, snapshot: "OrderedDict[str, Any]") -> Optional[Dict[str, Any]]:
        from ..fl.encrypted import train_encrypted

        to_train = self._policy(self.training_lower_bound_enc, self.training_upper_bound_enc, "first").select(snapshot)
        if not to_train:
            log.info("No behaviour defined for a number of workers less than " + str(self.training_lower_bound_enc))
            return None
        model = self._load_model()
        log.info("Distribute the data among the virtual workers...")
        result = train_encrypted(model, self._dataset(), list(to_train.keys()), self.args)
        save_model(model, self.path, meta={"model": self.args.model, "mode": "encrypted", "workers": list(to_train.keys())})
        self._deregister(to_train.keys())
        self.trainings_done += 1
        log.info("End encryption")
        return result

    # ------------------------------------------------------------------ remote mode
    async def training_remote(self, snapshot: "OrderedDict[str, Any]") -> Optional[Dict[str, Any]]:
        to_train = self._policy(self.training_lower_bound, self.training_upper_bound).select(snapshot)
        if not to_train:
            log.info("No behaviour defined for the number of devices achieved")
            return None
        model = self._load_model()
        if self.enabled_round > 1 and self.args.federate_after_n_batches < 0:
            log.info("Round activated!")
            self.args.set_federated_batches(ROUND_MODE_BATCHES)  # fc.py:533-535
        log.info("Federated batches: " + str(self.args.federate_after_n_batches))
        cfg = self._fit_config("remote")
        theta = flatten_params(model).cpu()
        loop = asyncio.get_running_loop()
        # one thread per selected device: every fit RPC of a round is in flight at the same time (the default
        # executor would cap the fan-out at min(32, cpu_count + 4) and serialise a 100-device round)
        from concurrent.futures import ThreadPoolExecutor
        pool = ThreadPoolExecutor(max_workers=max(1, len(to_train)), thread_name_prefix="fit-rpc")
        self.metrics.start_training(cfg.max_nr_batches)
        result: Dict[str, Any] = {"workers": list(to_train.keys()), "losses": {}, "rounds": self.enabled_round, "dropped": []}
        alive = OrderedDict(to_train)
        try:
            theta = await self._remote_rounds(alive, to_train, theta, cfg, loop, pool, model, result)
        finally:
            # whatever happened above, the devices' sockets are closed and they leave the registry (fc.py:573-580, 595-597)
            pool.shutdown(wait=False)
            for wid, worker in to_train.items():
                log.info("Closing socket for " + str(wid))
                self._close_quietly(worker)
            self._withdrawn.difference_update(to_train.keys())
            self._deregister(to_train.keys())
        unflatten_params(model, theta)
        save_model(model, self.path, meta={"model": self.args.model, "rounds": self.enabled_round, "workers": list(to_train.keys()), "mode": "remote"})
        eval_loss = None
        if self.evaluate_after:
            ds = self._dataset()
            from ..data import dataset_tensors
            x, y = dataset_tensors(ds, self.device)
            eval_loss = evaluate(model.to(self.device), x, y, verbose=False)["loss"]
            result["eval_loss"] = eval_loss
        self.metrics.end_training(eval_loss)
        self.trainings_done += 1
        return result

    async def _remote_rounds(self, alive, to_train, theta, cfg, loop, pool, model, result) -> torch.Tensor:
        """The round loop of ``training_remote`` (fc.py:540-568): fan the fit RPC out to every live device, FedAvg what came
        back, repeat.  Returns the final global parameters."""
        for r in range(self.enabled_round):
            log.info("\n\n#### ROUND {} #####".format(r))
            t0 = time.time()
            rcfg = FitConfig(**{**cfg.to_dict(), "seed": cfg.seed + r})

            async def one(wid: str, worker: RemoteWorkerClient):
                try:
                    fut = loop.run_in_executor(pool, lambda: worker.fit(theta, rcfg, timeout=self.fit_timeout))
                    flat, loss, n = await fut
                    # a device's reply is untrusted input: a wrong-length or non-finite model would poison (or abort) the
                    # whole average, so such a device counts as failed for this round
                    flat = torch.as_tensor(flat, dtype=torch.float32).reshape(-1)
                    if flat.numel() != theta.numel():
                        raise ValueError(f"model of {flat.numel()} parameters returned, expected {theta.numel()}")
                    if not bool(torch.isfinite(flat).all()):
                        raise ValueError("model with non-finite parameters returned")
                    return wid, flat, loss, n
                except Exception as e:  # noqa: BLE001 - a failing worker must not sink the round
                    log.info("Worker %s failed this round: %r", wid, e)
                    return wid, None, None, 0

            traffic = lambda w: (getattr(w, "bytes_sent", 0), getattr(w, "bytes_received", 0))  # noqa: E731 - any handle type
            sent0 = {wid: traffic(w) for wid, w in alive.items()}
            results = await asyncio.gather(*[one(wid, w) for wid, w in alive.items()])
            bytes_out = sum(traffic(w)[0] - sent0[wid][0] for wid, w in to_train.items() if wid in sent0)
            bytes_in = sum(traffic(w)[1] - sent0[wid][1] for wid, w in to_train.items() if wid in sent0)
            flats, counts, ids = [], [], []
            for wid, flat, loss, n in results:
                if flat is not None:
                    flats.append(flat)
                    counts.append(n)
                    ids.append(wid)
                    self.metrics.worker_loss(wid, loss)
                    result["losses"][wid] = loss
                else:
                    result["dropped"].append(wid)
                    alive.pop(wid, None)
            if flats:
                stacked = torch.stack(flats).to(self.device)
                w = normalized_weights(counts if self.args.weighted else None, len(flats), device=self.device)
                th = theta.to(self.device)
                ops.fedavg_apply(th, stacked, w, self.args.server_lr)
                theta = th.cpu()
                self._average_buffers(model, [getattr(alive.get(wid), "last_buffers", None) for wid in ids], w.cpu())
            # traffic of this round: model + fit config towards the devices, trained model + loss back (paper §4.3)
            self.metrics.end_round(r, time.time() - t0, selected=ids, n_k=counts, bytes_out=bytes_out, bytes_in=bytes_in)
            result["bytes_out"] = result.get("bytes_out", 0) + bytes_out
            result["bytes_in"] = result.get("bytes_in", 0) + bytes_in
            self._maybe_checkpoint(model, theta, r, {"workers": list(to_train.keys()), "mode": "remote"})
            if not alive:
                break
        return theta

    @staticmethod
    def _average_buffers(model, buffers, weights) -> None:
        """BatchNorm models in remote mode: the devices return their running statistics next to the parameters; the global
        model gets their FedAvg-weighted mean (PySyft's federated_avg averages parameters only — with it the reference could
        not train a BatchNorm model remotely at all; documented in docs/PARITY.md)."""
        mine = [b for b in model.buffers() if b.is_floating_point()]
        total = sum(b.numel() for b in mine)
        if not mine or any(b is None or b.numel() != total or not bool(torch.isfinite(b).all()) for b in buffers):
            return
        avg = (torch.stack([b.float() for b in buffers]) * weights.view(-1, 1).float()).sum(0)
        off = 0
        with torch.no_grad():
            for b in mine:
                b.copy_(avg[off:off + b.numel()].view_as(b).to(b.device))
                off += b.numel()

    # ------------------------------------------------------------------ inference (remote only)
    def _inference(self, worker: RemoteWorkerClient) -> None:
        model = self._load_model()
        flat = flatten_params(model)
        try:
            count = worker.search("inference")
            log.info("inference tensors found: %d", count)
            if count > 0:
                pred = worker.predict(flat, self.args.model)
                self.last_predictions = pred
                log.info(pred)
            else:
                log.info("Inference data not found!")
        finally:
            self.known_workers.pop(worker.id, None)
            worker.close()


# --------------------------------------------------------------------------------------------------
def train_virtual_workers(theta: torch.Tensor, model, fed, cfg: FitConfig, round_idx: int):
    """One round of local training for every virtual worker, each starting from ``theta``.

    On a GPU with a persistent kernel for the model (ops.persistent_path) all K workers train **concurrently in one
    launch** (one CTA or one cluster per worker); otherwise they run one after the other through ``local_fit``.
    Returns ``(flats[K,P], last_losses[K], sample_counts[K])``.
    """
    k = len(fed.workers)
    device = theta.device
    flats = theta.unsqueeze(0).repeat(k, 1).contiguous()
    counts = [len(fed[w]) for w in fed.workers]
    losses = [0.0] * k
    spec = model.spec if isinstance(model, MLPNet) else None
    fused = (spec is not None and device.type == "cuda"
             and ops.persistent_path(spec.dims, spec.out_activation, cfg.batch_size, resolve_loss(cfg.model, cfg.loss), device))
    if fused:
        loss_out = torch.zeros(k, 2, device=device)
        tasks, idx = [], []
        for i, wid in enumerate(fed.workers):
            sh = fed[wid]
            if len(sh) == 0:
                continue
            perm = make_perm(len(sh), FitConfig(**{**cfg.to_dict(), "seed": cfg.seed + 31 * i}), device, round_idx)
            x = sh.x.view(len(sh), -1).contiguous().float()
            y = sh.y.contiguous().float().view(len(sh), -1)
            tasks.append(ops.ClientTask(x=x, y=y, theta_in=theta, theta_out=flats[i], perm=perm, loss_out=loss_out[i]))
            idx.append(i)
        if tasks:
            descs = ops.build_client_descs(tasks, device)
            ops.mlp_local_sgd_multi(spec.dims, spec.out_activation, descs, len(tasks), cfg.batch_size, cfg.lr,
                                    cfg.epochs, cfg.max_nr_batches, resolve_loss(cfg.model, cfg.loss))
            vals = loss_out[:, 0].tolist()
            for i in idx:
                losses[i] = vals[i]
        return flats, losses, counts
    if spec is not None and device.type == "cpu" and ops.host.available() and spec.out_activation in ("none", "sigmoid"):
        # CPU box: the native host executor trains the K workers concurrently on K threads (ops/csrc/mlp_host.cpp)
        idx = [i for i, wid in enumerate(fed.workers) if len(fed[wid]) > 0]
        if idx:
            shards = [fed[fed.workers[i]] for i in idx]
            perms = [make_perm(len(sh), FitConfig(**{**cfg.to_dict(), "seed": cfg.seed + 31 * i}), device, round_idx)
                     for i, sh in zip(idx, shards)]
            res = ops.host.mlp_local_sgd_multi(spec.dims, spec.out_activation, [flats[i] for i in idx], [sh.x for sh in shards],
                                               [sh.y for sh in shards], perms, cfg.batch_size, cfg.lr, cfg.epochs,
                                               cfg.max_nr_batches, resolve_loss(cfg.model, cfg.loss))
            for j, i in enumerate(idx):
                losses[i] = float(res[j, 0])
        return flats, losses, counts
    for i, wid in enumerate(fed.workers):
        sh = fed[wid]
        if len(sh) == 0:
            continue
        wcfg = FitConfig(**{**cfg.to_dict(), "seed": cfg.seed + 31 * i})
        last, _ = local_fit(flats[i], model, sh.x, sh.y, wcfg, round_idx)
        losses[i] = float(last)
    return flats, losses, counts

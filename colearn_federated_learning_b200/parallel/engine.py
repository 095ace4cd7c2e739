"""FederatedEngine — the round loop of the reference mapped onto the GPUs of one box.

One process per GPU.  Rank ``coordinator_rank`` (0) hosts the coordinator role *and* is a worker
(co-located, SURVEY §7.0); every rank holds a private shard.  One **round** is what the
reference's ``training_remote`` loop body does (``federated_coordinator.py:540-568``):

    broadcast θ to the selected workers      train_config.send(worker)      cf.py:209   (K1)
    each worker: local SGD on its shard      worker.async_fit(...)          cf.py:210   (K12)
    gather the trained models                model_ptr.get()                cf.py:211   (K2)
    θ ← FedAvg (uniform or n_k-weighted)     utils.federated_avg(models)    fc.py:568   (K3)

Backends
  ``fused``  hand-written kernels over symmetric memory, **no NCCL on the round path**:
             * ``star``    (persistent-MLP models): the worker kernel waits for the broadcast flag,
               trains, writes ``w_k·θ_k`` straight into the coordinator's slot over NVLink and
               raises an arrive flag; ONE coordinator kernel then reduces + applies + pushes the
               next round's θ into every selected inbox.  2 launches/round on rank 0, 1 elsewhere.
             * ``twoshot`` (large models): in-place symmetric all-reduce-with-apply on the work
               arenas (``twoshot_fedavg_kernel``), dual fp32 + bf16 write, per-chunk ready flags.
  ``cpu``    gloo + ``ops.reference`` — same semantics, for tests on a GPU-less box.
The ``nccl`` comparator lives in ``baseline/`` and shares none of this code.
"""
from __future__ import annotations

import logging
import os
import time
from dataclasses import dataclass, field
from typing import Any, Dict, List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist
import torch.nn as nn

from .. import ops
from ..fl.fedavg import normalized_weights
from ..fl.trainer import FitConfig, local_fit, resolve_loss
from ..models import MLPNet, build_model, flatten_params, num_params, state_dict_from_flat
from ..utils.checkpoint import save_state_dict
from ..utils.tracing import PhaseTimer, nvtx_range

log = logging.getLogger(__name__)


def _dist_ready() -> bool:
    return dist.is_available() and dist.is_initialized()


@dataclass
class RoundReport:
    rounds: int
    world: int
    backend: str
    algo: str
    device_ms: float                      # CUDA-event time of the whole call on this rank
    losses: Optional[torch.Tensor] = None  # [rounds, world, 2] (coordinator) last/mean loss per worker
    launches: int = 0                      # kernels of this repo launched inside the timed region
    bytes_bcast: int = 0
    bytes_reduce: int = 0
    extra: Dict[str, Any] = field(default_factory=dict)


class FederatedEngine:
    def __init__(self, model: str = "mlp", *, backend: str = "auto", device: Optional[torch.device] = None,
                 group: Optional[dist.ProcessGroup] = None, batch_size: int = 1, lr: float = 0.01,
                 local_epochs: int = 1, max_batches: int = -1, loss: str = "auto", weighted: bool = True,
                 server_lr: float = 1.0, coordinator_rank: int = 0, algo: str = "auto", seed: int = 1,
                 shuffle: bool = True, chunk_elems: int = 0, bf16_shadow: bool = False,
                 round_deadline_ms: float = 0.0, clients_per_rank: int = 1,
                 model_kwargs: Optional[Dict[str, Any]] = None, overlap_reduce: Optional[bool] = None,
                 phase_timing: Optional[bool] = None) -> None:
        self.rank = dist.get_rank(group) if _dist_ready() else 0
        self.world = dist.get_world_size(group) if _dist_ready() else 1
        self.group = group
        self.coord = coordinator_rank
        if device is None:
            if torch.cuda.is_available():
                device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", self.rank % max(1, torch.cuda.device_count()))))
            else:
                device = torch.device("cpu")
        self.device = torch.device(device)
        if backend == "auto":
            backend = "fused" if self.device.type == "cuda" else "cpu"
        if backend == "fused" and self.device.type != "cuda":
            raise RuntimeError("backend 'fused' needs a CUDA device")
        self.backend = backend
        self.model_name = model
        torch.manual_seed(seed)  # identical init on every rank (only the coordinator's copy matters)
        self.model: nn.Module = build_model(model, **(model_kwargs or {}))
        self.spec = self.model.spec if isinstance(self.model, MLPNet) else None
        self.P = num_params(self.model)
        self.P4 = (self.P + 3) // 4 * 4
        self.cfg = FitConfig(model=model, loss=resolve_loss(model, loss), batch_size=batch_size, epochs=local_epochs,
                             max_nr_batches=max_batches, lr=lr, shuffle=shuffle, seed=seed)
        self.weighted = weighted
        self.server_lr = server_lr
        self.seed = seed
        # a specialised persistent kernel, or (CUDA, batch <= ops.GENERIC_MAX_BATCH) the generic one
        persistent = self.spec is not None and ops.persistent_path(self.spec.dims, self.spec.out_activation, batch_size,
                                                                   self.cfg.loss, self.device)
        if algo == "auto":
            algo = "star" if persistent else "twoshot"
        if algo == "star" and backend == "fused" and not persistent:
            raise ValueError(f"algo 'star' needs a persistent-kernel model, got {model}")
        self.algo = algo
        if not chunk_elems:
            # flag/work granularity of the two-shot kernel: >= ~2 CTAs per SM worth of chunks per rank
            target = max(1, self.P4 // (self.world * 296))
            chunk_elems = 2048
            while chunk_elems < target and chunk_elems < 65536:
                chunk_elems *= 2
        self.chunk_elems = int(chunk_elems)
        self.bf16_shadow = bf16_shadow
        # failure detection: a selected worker that has not delivered within this many ms of the coordinator
        # starting its reduce is dropped from that round (its weight is renormalised away); 0 = wait forever
        self.round_deadline_ms = float(round_deadline_ms)
        # many virtual clients (federated devices) per GPU: one CTA each, summed locally before the NVLink push
        self.clients_per_rank = max(1, int(clients_per_rank))
        self.use_graphs = os.environ.get("COLEARN_CUDA_GRAPHS", "1") != "0"
        # multimem.ld_reduce / multimem.st in the two-shot kernel.  Through the switch every GPU sends its whole vector once (each
        # element is pulled by its owner's ld_reduce) plus its reduced share once, and receives the same: (1 + 1/W) x model bytes
        # per direction, against 2 (W-1)/W x for peer loads + peer stores.  The GPUs' own NVLink counters agree (profiles/
        # r2_nvlink_counters.json: W=2 1.50 x vs 1.00 x, and 0.57 vs 0.36 ms for 201 MB), so "auto" takes the switch from W = 4 up
        nvls_env = os.environ.get("COLEARN_NVLS", "auto")
        self.use_nvls = nvls_env == "1" or (nvls_env not in ("0", "1") and self.world >= 4)
        # fused wgrad GEMM -> FedAvg reduce (ops/produced.py, opt-in until measured): the two-shot kernel runs on
        # `overlap_ctas` CTAs NEXT TO the last local backward pass and reduces chunks as the wgrad epilogues report them
        if overlap_reduce is None:
            overlap_reduce = os.environ.get("COLEARN_OVERLAP_REDUCE", "0") == "1"
        self.overlap_reduce = bool(overlap_reduce) and algo == "twoshot" and backend == "fused"
        self.overlap_ctas = max(1, int(os.environ.get("COLEARN_OVERLAP_CTAS", "16")))
        self.overlap_timeout_s = float(os.environ.get("COLEARN_OVERLAP_TIMEOUT_S", "20"))
        # per-phase device timing (SURVEY §5): CUDA-event pairs around the H2D copy / broadcast / local fit / reduce+apply /
        # read-back launches of every round, reported as RoundReport.extra["phases_ms"]; the NVTX ranges of the same phases
        # (COLEARN_NVTX=1) are always in place.  Off by default: the event records cost ~1 us each on the 20 kB-model rounds.
        if phase_timing is None:
            phase_timing = os.environ.get("COLEARN_PHASE_TIMING", "0") == "1"
        self.phase_timing = bool(phase_timing)
        self.epoch = 0          # monotonically increasing flag epoch (never reset)
        self.rounds_done = 0
        self.x: Optional[torch.Tensor] = None
        self.y: Optional[torch.Tensor] = None
        self.n_local = 0
        self.counts: List[int] = [0] * self.world
        self._stream_inputs: Optional[Tuple[torch.Tensor, torch.Tensor]] = None
        if backend == "fused":
            self._init_fused()
        else:
            self.theta = flatten_params(self.model).to(self.device)
        self.model.to(self.device)

    # ------------------------------------------------------------------------------------------
    def _init_fused(self) -> None:
        from .symm import SymmetricArena

        torch.cuda.set_device(self.device)
        W, P4 = self.world, self.P4
        if self.algo == "star":
            layout = {"inbox": (P4, torch.float32), "slots": (W * P4, torch.float32), "flags": (64, torch.int32),
                      "losses": (2 * W, torch.float32)}
        else:
            self.n_chunks = (P4 + self.chunk_elems - 1) // self.chunk_elems
            layout = {"work": (P4, torch.float32), "chunk_flags": (self.n_chunks, torch.int32),
                      "flags": (64, torch.int32), "losses": (2 * W, torch.float32)}
            if self.bf16_shadow:
                layout["shadow"] = (P4, torch.bfloat16)
            if self.overlap_reduce:
                layout["produced"] = (W * self.n_chunks, torch.int32)   # [producer rank, chunk] epochs of the chunks I own
            if self.round_deadline_ms > 0:
                # failure detection on the two-shot path: the coordinator's arrived-set decisions (ring of 8 x {epoch, mask}) and
                # a second arena that also receives every round's result — a rank that missed a deadline trained in place on a work
                # arena the owners overwrote under it and restores it from there (comm.cu: twoshot_resync_kernel)
                layout["decision"] = (16, torch.int32)
                layout["global"] = (P4, torch.float32)
        self.arena = SymmetricArena(layout, self.device, self.group)
        self.ext = ops._ext.require()
        # every cross-GPU flag wait of the round kernels is bounded: past this many seconds without the peer's signal the
        # kernel traps and the round raises instead of hanging the box (0 = wait forever)
        self.spin_timeout_s = float(os.environ.get("COLEARN_SPIN_TIMEOUT_S", "120"))
        self.ext.set_spin_limit(self.spin_timeout_s)
        self.grid_counter = torch.zeros(4, dtype=torch.int32, device=self.device)
        self.decision = torch.zeros(2, dtype=torch.int32, device=self.device)
        self.epoch_dev = torch.zeros(1, dtype=torch.int32, device=self.device)
        flat = flatten_params(self.model).to(self.device)
        if self.algo == "star":
            self.theta = torch.zeros(P4, device=self.device)
            self.theta[: self.P].copy_(flat)
        else:
            self.theta = self.arena.tensor("work")
            self.theta[: self.P].copy_(flat)
            self.weights_dev = torch.zeros(16, device=self.device)
            if self.world > 1:
                # initial model sync: every rank pulls the coordinator's arena over NVLink
                torch.cuda.synchronize(self.device)
                dist.barrier(group=self.group)
                if self.rank != self.coord:
                    self.ext.p2p_copy(self.arena.ptr("work"), self.arena.ptr("work", self.coord), P4, 0, 0, 296)
                torch.cuda.synchronize(self.device)
                dist.barrier(group=self.group)
        self.loss_host = torch.zeros(2 * W, dtype=torch.float32).pin_memory()
        if self.algo == "star" and self.clients_per_rank > 1:
            C = self.clients_per_rank
            self.client_slots = torch.zeros(C, P4, device=self.device)
            self.client_losses = torch.zeros(C, 2, device=self.device)
            self.push_counter = torch.zeros(1, dtype=torch.int32, device=self.device)

    # ------------------------------------------------------------------------------------------
    def set_local_data(self, x: torch.Tensor, y: torch.Tensor) -> None:
        """Attach this rank's private shard (device-resident from here on)."""
        self.x = x.to(self.device).float().contiguous()
        yy = y.to(self.device).float()
        self.y = (yy.view(-1, 1) if yy.dim() == 1 else yy).contiguous()
        self.n_local = int(self.x.shape[0])
        if _dist_ready() and self.world > 1:
            gathered = [0] * self.world
            dist.all_gather_object(gathered, self.n_local, group=self.group)
            self.counts = [int(c) for c in gathered]
        else:
            self.counts = [self.n_local]

    def load_global(self, flat: torch.Tensor) -> None:
        self.theta[: self.P].copy_(flat.to(self.device).float().reshape(-1)[: self.P])

    def global_flat(self) -> torch.Tensor:
        return self.theta[: self.P]

    def global_state_dict(self):
        return state_dict_from_flat(self.model, self.global_flat())

    def save_checkpoint(self, path: str) -> Optional[str]:
        if self.rank != self.coord:
            return None
        return save_state_dict(self.global_state_dict(), path,
                               meta={"rounds": self.rounds_done, "world": self.world, "model": self.model_name,
                                     "backend": self.backend, "algo": self.algo, "sample_counts": self.counts})

    # ------------------------------------------------------------------------------------------
    def _round_weights(self, mask: int) -> List[float]:
        sel = [k for k in range(self.world) if (mask >> k) & 1]
        if not sel:
            return [0.0] * self.world
        w = normalized_weights([self.counts[k] for k in sel] if self.weighted else None, len(sel))
        out = [0.0] * self.world
        for k, v in zip(sel, w.tolist()):
            out[k] = v
        return out

    def _masks(self, rounds: int, masks) -> List[int]:
        full = (1 << self.world) - 1
        if masks is None:
            return [full] * rounds
        if isinstance(masks, int):
            return [masks & full] * rounds
        assert len(masks) == rounds
        return [int(m) & full for m in masks]

    def run_rounds(self, rounds: int, masks=None, host_inputs: Optional[Sequence[Tuple[torch.Tensor, torch.Tensor]]] = None,
                   read_back=False, barrier: bool = True) -> RoundReport:
        """Run ``rounds`` federated rounds.  ``masks``: selection bitmask(s) (bit k = rank k
        trains).  ``host_inputs``: per-round pinned-host ``(x, y)`` for this rank, copied H2D
        inside the round (end-to-end mode); ``read_back`` additionally copies each round's losses
        D2H and synchronises per round; ``read_back="pipelined"`` (star path) still copies every round's
        losses D2H but lets the host read them one round late (``loss_history``), so the GPU does not wait for the host.  ``barrier=False`` skips the host-side process-group
        barriers around the timed region (rounds are self-synchronising through device flags)."""
        self._barrier = barrier
        if self.x is None and host_inputs is None:
            raise RuntimeError("set_local_data() first")
        ms = self._masks(rounds, masks)
        if self.backend == "cpu":
            return self._run_cpu(rounds, ms)
        if self.algo == "star":
            return self._run_star(rounds, ms, host_inputs, read_back)
        return self._run_twoshot(rounds, ms, host_inputs, read_back)

    def _align_streams(self) -> None:
        """Device-side barrier behind the host-side one (``barrier=True`` calls only): every rank raises its slot of an
        alignment row in every peer's flag block (``signal_peers_kernel``) and waits for the whole row in its own
        (``wait_flags_kernel``).  Processes leave ``dist.barrier`` tens of microseconds apart; a rank that leaves early would
        otherwise count its wait for the coordinator's first launch as round time (max-over-ranks event timing of a sub-ms
        round).  Outside every timed region: the events are recorded after it."""
        if self.backend != "fused" or self.world <= 1 or self.world > 16:
            return
        self._align_seq = getattr(self, "_align_seq", 0) + 1
        arena, r = self.arena, self.rank
        self.ext.signal_peers([arena.ptr("flags", k, 32 + r) for k in range(self.world)], self._align_seq)
        self.ext.wait_flags(arena.ptr("flags", None, 32), self.world, self._align_seq)

    # ------------------------------------------------------------------------------------------ tracing
    def _phase(self, name: str):
        """Context manager around the launches of one phase of a round: NVTX range + (with ``phase_timing``) an event pair."""
        timer = getattr(self, "_phases", None)
        return timer.phase(name) if timer is not None else nvtx_range(name)

    def _phases_begin(self) -> None:
        self._phases = PhaseTimer(self.device) if self.phase_timing else None

    def _phases_end(self) -> Optional[Dict[str, float]]:
        timer, self._phases = getattr(self, "_phases", None), None
        return {k: round(v, 4) for k, v in timer.summary().items()} if timer is not None else None

    # ------------------------------------------------------------------------------------------ self check
    def verify_round(self, mask: Optional[int] = None) -> Dict[str, Any]:
        """Run ONE more round twice on the same inputs — through the fused path, and with ``dist.broadcast`` + the same local
        fit + ``dist.reduce`` (NCCL) + a host-side apply — and report the difference on the coordinator.  The local fits are
        bit-identical (same kernel, same sample order), so what is compared is the communication: broadcast, per-worker
        ``n_k`` scale, selection mask, reduce order, server apply.  ``star`` path only (``{"skipped": ...}`` otherwise)."""
        if self.backend != "fused" or self.algo != "star" or self.clients_per_rank != 1:
            return {"skipped": f"verify_round covers the fused star path with one client per rank (algo={self.algo})"}
        W, r, dev, cfg = self.world, self.rank, self.device, self.cfg
        full = (1 << W) - 1
        mask = full if mask is None else (int(mask) & full)
        theta0 = self.theta[: self.P].clone()
        if _dist_ready() and W > 1:
            dist.broadcast(theta0, src=self.coord, group=self.group)                     # K1, library form
        w = self._round_weights(mask)[r]
        contrib = torch.zeros_like(theta0)
        if (mask >> r) & 1:
            local = theta0.clone()
            perm = None
            if cfg.shuffle:
                pseed = ((self.seed * 1000003 + 17 * r + 1) & 0x7FFFFFFFFFFF) | 1
                row0 = self.rounds_done * cfg.epochs
                perm = ops.device_permutation(self.n_local, row0 + cfg.epochs, pseed, dev)[row0:].contiguous()
            ops.mlp_local_sgd(local, self.spec.dims, self.x, self.y, perm, cfg.batch_size, cfg.lr, cfg.epochs, cfg.max_nr_batches,
                              cfg.loss, self.spec.out_activation)
            contrib = local * w
        if _dist_ready() and W > 1:
            dist.reduce(contrib, dst=self.coord, group=self.group)                       # K2 + K3, library form
        expected = theta0 + self.server_lr * (contrib - theta0)
        rep = self.run_rounds(1, masks=mask)
        got = self.theta[: self.P]
        out: Dict[str, Any] = {"algo": self.algo, "provider": rep.extra.get("provider"), "multicast": rep.extra.get("multicast"),
                               "mask": mask, "world": W}
        if r == self.coord:
            err = float((got - expected).abs().max())
            ref = float(expected.abs().max())
            out.update(max_abs_err=err, max_abs_ref=ref, rel_err=err / max(ref, 1e-30), moved=float((got - theta0).abs().max()),
                       ok=bool(err <= 1e-5 * max(ref, 1.0) and torch.isfinite(got).all()))
        return out

    # ------------------------------------------------------------------------------------------ star
    def _run_star(self, rounds: int, masks: List[int], host_inputs, read_back: bool) -> RoundReport:
        ext, arena, W, P4, r = self.ext, self.arena, self.world, self.P4, self.rank
        dev = self.device
        cfg = self.cfg
        n = self.n_local if host_inputs is None else int(host_inputs[0][0].shape[0])
        if host_inputs is not None and (self.x is None or self.x.shape[0] != n):
            self.x = torch.empty(n, host_inputs[0][0].shape[1], device=dev)
            self.y = torch.empty(n, 1, device=dev)
            self.set_local_data(self.x, self.y)
        e0 = self.epoch
        coord_slots = arena.ptr("slots", self.coord, r * P4)
        coord_loss = arena.ptr("losses", self.coord, 2 * r)
        coord_arrive = arena.ptr("flags", self.coord, 1 + r)
        C = self.clients_per_rank
        # Single-round calls (the e2e / per-step usage) reuse a cached plan: the descriptors of the next kPlanRounds rounds
        # are packed once; a call then costs no descriptor packing and no H2D of descriptors (the shuffle itself happens
        # inside the worker kernel).  Epochs advance by 2 per single-round call (broadcast, then reduce without broadcast).
        kPlanRounds = 256
        plan_key = (masks[0], n, self.x.data_ptr(), cfg.batch_size, cfg.epochs, cfg.max_nr_batches, cfg.lr, C)
        plan = getattr(self, "_star_plan", None)
        cached = (rounds == 1 and plan is not None and plan["key"] == plan_key and plan["used"] < plan["cap"]
                  and plan["e0"] + 2 * plan["used"] == e0)
        if cached:
            descs, desc_base = plan["descs"], plan["used"] * C
            plan["used"] += 1
        else:
            cap = kPlanRounds if rounds == 1 else rounds
            stride = 2 if rounds == 1 else 1
            # sample order: the worker kernel tabulates the keyed Feistel permutation of its epochs itself, before it waits for
            # the round's broadcast (ClientDesc::perm_seed / perm_row0 / perm_scratch) — a round's shuffle costs no launch and is
            # inside whatever region times the round; round i, epoch e uses row (rounds_done + i) * epochs + e of the client's key
            pseed = ((self.seed * 1000003 + 17 * r + 1) & 0x7FFFFFFFFFFF) | 1 if cfg.shuffle else 0
            tasks = []
            if C > 1:
                from ..data import shard_bounds
                cb = [b for b in shard_bounds(n, C)]
            # scratch of the kernel-made permutation tables: [epochs, n_client] ints per client, reused every round
            sizes_c = [n] if C == 1 else [hi - lo for lo, hi in cb]
            key_s = (tuple(sizes_c), cfg.epochs)
            if pseed and getattr(self, "_perm_scratch_key", None) != key_s:
                self._perm_scratch = [torch.empty(max(1, cfg.epochs * max(1, m)), dtype=torch.int32, device=dev) for m in sizes_c]
                self._perm_scratch_key = key_s
            for i in range(cap):
                w = self._round_weights(masks[i] if rounds > 1 else masks[0])[r]
                row0 = (self.rounds_done + i) * cfg.epochs
                ev = e0 + stride * i + 1
                if C == 1:
                    tasks.append(ops.ClientTask(x=self.x, y=self.y, theta_in=arena.ptr("inbox"), theta_out=coord_slots,
                                                perm_seed=pseed, perm_row0=row0, perm_scratch=self._perm_scratch[0] if pseed else None,
                                                loss_out=coord_loss, wait_flag=arena.ptr("flags"), wait_value=ev,
                                                signal_flag=coord_arrive, signal_value=ev, out_scale=w))
                else:
                    # C virtual clients on this GPU (one CTA each); each starts from the broadcast theta, trains on its
                    # contiguous sub-shard and leaves w_rank * (n_c / n_rank) * theta_c in a local slot
                    for c, (lo, hi) in enumerate(cb):
                        share = ((hi - lo) / max(1, n)) if self.weighted else 1.0 / C
                        tasks.append(ops.ClientTask(x=self.x[lo:hi], y=self.y[lo:hi], theta_in=arena.ptr("inbox"),
                                                    theta_out=self.client_slots[c],
                                                    perm_seed=(pseed + 2 * 7919 * (c + 1)) if pseed else 0, perm_row0=row0,
                                                    perm_scratch=self._perm_scratch[c] if pseed else None,
                                                    loss_out=self.client_losses[c],
                                                    wait_flag=arena.ptr("flags"), wait_value=ev, out_scale=w * share))
            descs = ops.build_client_descs(tasks, dev)
            desc_base = 0
            if rounds == 1:
                self._star_plan = {"key": plan_key, "descs": descs, "cap": cap, "used": 1, "e0": e0}
        inbox_ptrs = arena.peer_ptrs("inbox")
        bflag_ptrs = arena.peer_ptrs("flags")
        n_blocks = max(1, min(148, (P4 // 4 + 255) // 256))
        is_coord = r == self.coord
        # every row of losses_log is overwritten by the round's copy; arrived_log is only read in deadline mode: no fill
        # launches in front of the round's first kernel (single-round calls pay them every call)
        losses_log = torch.empty(rounds, W, 2, device=dev) if is_coord else None
        arrived_log = (torch.zeros(rounds, dtype=torch.int32, device=dev) if self.round_deadline_ms > 0
                       else torch.empty(rounds, dtype=torch.int32, device=dev))
        launches = 0
        if _dist_ready() and W > 1 and self._barrier:
            dist.barrier(group=self.group)
            self._align_streams()
        torch.cuda.synchronize(dev)
        if getattr(self, "_star_events", None) is None:
            self._star_events = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        ev0, ev1 = self._star_events
        ev0.record()
        # read_back="pipelined": every round's losses are still copied to the host, but the host reads them one round late
        pipelined = read_back == "pipelined"
        if pipelined:
            if getattr(self, "loss_ring", None) is None:
                self.loss_ring = torch.zeros(2, 2 * W, dtype=torch.float32).pin_memory()
                self._ring_ev = (torch.cuda.Event(), torch.cuda.Event())
            ring_ev = self._ring_ev
            self.loss_history: List[torch.Tensor] = []

        def star(do_reduce: bool, do_bcast: bool, mask_reduce: int, mask_bcast: int, arrive_epoch: int, bcast_epoch: int):
            wts = [float(v) for v in self._round_weights(mask_reduce)] if do_reduce else [0.0] * W
            # reduce over the workers of the finished round, broadcast to those of the next one
            if do_reduce and do_bcast and mask_reduce != mask_bcast:
                ext.star_round(self.theta.data_ptr(), arena.ptr("slots"), P4, arena.ptr("flags", None, 1), arrive_epoch,
                               inbox_ptrs, bflag_ptrs, bcast_epoch, 0, mask_reduce, self.server_lr, P4, True, False,
                               self.grid_counter.data_ptr(), n_blocks, self.round_deadline_ms, wts, self.decision.data_ptr())
                ext.star_round(self.theta.data_ptr(), arena.ptr("slots"), P4, arena.ptr("flags", None, 1), arrive_epoch,
                               inbox_ptrs, bflag_ptrs, bcast_epoch, arena.mc_ptr("inbox"),
                               mask_bcast, self.server_lr, P4, False, True, self.grid_counter.data_ptr(), n_blocks, 0.0, wts, 0)
                return 2
            mask = mask_reduce if do_reduce else mask_bcast
            # NVLS broadcast also for a subset: multimem.st lands in every rank's inbox (one egress copy, the switch replicates);
            # only the selected ranks get their flag raised, the others never look at theirs
            mc = arena.mc_ptr("inbox") if do_bcast else 0
            ext.star_round(self.theta.data_ptr(), arena.ptr("slots"), P4, arena.ptr("flags", None, 1), arrive_epoch,
                           inbox_ptrs, bflag_ptrs, bcast_epoch, mc, mask, self.server_lr, P4, do_reduce, do_bcast,
                           self.grid_counter.data_ptr(), n_blocks, self.round_deadline_ms if do_reduce else 0.0, wts,
                           self.decision.data_ptr())
            return 1

        self._phases_begin()
        if is_coord:
            with self._phase("bcast"):
                launches += star(False, True, 0, masks[0], 0, e0 + 1)
        for i in range(rounds):
            if host_inputs is not None:
                with self._phase("h2d"):
                    hx, hy = host_inputs[i]
                    self.x.copy_(hx, non_blocking=True)
                    self.y.copy_(hy.view(-1, 1), non_blocking=True)
            if (masks[i] >> r) & 1:
                with self._phase("local_fit"):
                    ops.mlp_local_sgd_multi(self.spec.dims, self.spec.out_activation, descs, C, cfg.batch_size, cfg.lr,
                                            cfg.epochs, cfg.max_nr_batches, cfg.loss, desc_offset=desc_base + i * C)
                    launches += 1
                    if C > 1:
                        ext.reduce_push(self.client_slots.data_ptr(), C, P4, P4, coord_slots, self.client_losses.data_ptr(),
                                        coord_loss, coord_arrive, e0 + i + 1, self.push_counter.data_ptr(), n_blocks)
                        launches += 1
            if is_coord:
                last = i == rounds - 1
                with self._phase("reduce_apply" if last else "reduce_apply_bcast"):
                    launches += star(True, not last, masks[i], masks[i + 1] if not last else 0, e0 + i + 1, e0 + i + 2)
                losses_log[i].copy_(arena.tensor("losses").view(W, 2), non_blocking=True)
                if self.round_deadline_ms > 0:
                    arrived_log[i].copy_(self.decision[1], non_blocking=True)
                if pipelined:
                    # lagged read-back: round i's losses go to pinned slot i % 2; the host waits for round i-1's copy only
                    # after round i is enqueued, so the GPU never idles behind the host
                    slot = i & 1
                    self.loss_ring[slot].copy_(arena.tensor("losses"), non_blocking=True)
                    ring_ev[slot].record()
                    if i >= 1:
                        ring_ev[1 - slot].synchronize()
                        self.loss_history.append(self.loss_ring[1 - slot].clone())
                elif read_back:
                    self.loss_host.copy_(arena.tensor("losses"), non_blocking=True)
                    torch.cuda.current_stream(dev).synchronize()
            elif pipelined:
                ring_ev[i & 1].record()
                if i >= 1:
                    ring_ev[1 - (i & 1)].synchronize()        # bound the run-ahead of a worker rank to one round
            elif read_back:
                torch.cuda.current_stream(dev).synchronize()
        if pipelined and rounds > 0:
            ring_ev[(rounds - 1) & 1].synchronize()
            if is_coord:
                self.loss_history.append(self.loss_ring[(rounds - 1) & 1].clone())
                self.loss_host.copy_(self.loss_history[-1])
        ev1.record()
        torch.cuda.synchronize(dev)
        phases = self._phases_end()
        self.epoch = e0 + rounds + 1
        self.rounds_done += rounds
        if _dist_ready() and W > 1 and self._barrier:
            dist.barrier(group=self.group)
        nsel = [bin(m).count("1") for m in masks]
        return RoundReport(rounds, W, "fused", "star", ev0.elapsed_time(ev1), losses_log, launches,
                           bytes_bcast=4 * self.P * sum(nsel), bytes_reduce=4 * self.P * sum(nsel),
                           extra={"provider": arena.provider, "multicast": arena.has_multicast, "phases_ms": phases,
                                  "arrived_masks": arrived_log.tolist() if (is_coord and self.round_deadline_ms > 0) else None})

    # ------------------------------------------------------------------------------------------ twoshot
    def _layerwise_trainer(self):
        """tcgen05 layer-wise trainer bound to the work arena (+ bf16 shadow arena), or None."""
        if getattr(self, "_lw_checked", False):
            return self._lw
        self._lw_checked, self._lw = True, None
        if self.spec is not None:
            from ..fl.layerwise import LayerwiseMLPTrainer
            if LayerwiseMLPTrainer.supports_fused(self.spec, self.cfg):
                shadow = self.arena.tensor("shadow") if self.bf16_shadow else None
                self._lw = LayerwiseMLPTrainer(self.spec, self.theta[: self.P], self.cfg.batch_size, shadow=shadow)
        return self._lw

    def _produced_spec(self):
        """:class:`ops.produced.ProducedSpec` of this rank (fused wgrad -> reduce), or None when the mode is off / unusable."""
        if not self.overlap_reduce or self._layerwise_trainer() is None:
            return None
        if getattr(self, "_prod", None) is None:
            from ..ops.produced import ProducedSpec
            sms = torch.cuda.get_device_properties(self.device).multi_processor_count
            self.prod_count = torch.zeros(self.n_chunks, dtype=torch.int32, device=self.device)
            self.comm_stream = torch.cuda.Stream(device=self.device)
            self._prod = ProducedSpec.device(self.ext, self.prod_count, self.arena.peer_ptrs("produced"), self.epoch_dev, 1,
                                             chunk_elems=self.chunk_elems, n=self.P4, rank=self.rank,
                                             max_ctas=max(8, sms - self.overlap_ctas))
        return self._prod

    def _local_train_inplace(self, round_idx: int, epoch: int, produced=None, overlapped=None) -> torch.Tensor:
        """Local fit in place on the work arena.  Wide MLPs: tcgen05 layer-wise trainer whose first
        forward GEMMs consume the previous round's broadcast chunk by chunk (flags of ``epoch-1``);
        everything else: torch autograd (cuDNN convs) + this repo's loss / SGD kernels.

        ``produced`` / ``overlapped`` (fused wgrad -> FedAvg reduce): the last backward reports what it finalises and
        ``overlapped()`` — the launch of the two-shot kernel on the side stream — runs right before it is queued."""
        flat = self.theta[: self.P]
        lw = self._layerwise_trainer()
        if lw is None:
            if epoch > 1:
                self.ext.wait_flags(self.arena.ptr("chunk_flags"), self.n_chunks, epoch - 1)
            last, path = local_fit(flat, self.model, self.x, self.y, FitConfig(**{**self.cfg.to_dict()}), round_idx)
            from ..fl import trainer as _trainer
            self._last_path, self._train_launches = path, _trainer.LAST_FIT_LAUNCHES
            return last
        from ..fl.layerwise import ReadySpec
        from ..fl.trainer import make_perm
        n = self.x.shape[0]
        perm = make_perm(n, self.cfg, self.device, round_idx)
        cf_ptr = self.arena.ptr("chunk_flags")
        fused = epoch > 1 and self.bf16_shadow
        xs = self.x.view(n, -1)
        if fused and self.use_graphs and n % self.cfg.batch_size == 0:
            # launch-bound inner loop -> ONE CUDA-graph replay per round (flag epoch + sample order are device-side)
            if getattr(lw, "graph", None) is None:
                steps = (n // self.cfg.batch_size) * self.cfg.epochs
                if self.cfg.max_nr_batches and self.cfg.max_nr_batches > 0:
                    steps = min(steps, self.cfg.max_nr_batches)
                self.ext.set_flag(self.epoch_dev.data_ptr(), epoch - 1)
                lw.build_round_graph(flat, xs, self.y, self.cfg.lr, steps,
                                     ReadySpec(cf_ptr, self.chunk_elems, 0, self.epoch_dev.data_ptr()), self.n_chunks,
                                     produced=self._produced_spec())
            self.ext.set_flag(self.epoch_dev.data_ptr(), epoch - 1)
            if produced is None and getattr(lw, "graph_tail", None) is not None:
                # a round without the overlap (partial selection) on a trainer captured for it: the reports are made anyway
                # (counters return to zero, the tables are simply not read); the classic two-shot follows in stream order
                overlapped = None
            last = lw.run_round_graph(perm, n, between=overlapped)
            self._last_path = "layerwise+fused_bcast+cuda_graph" + ("+overlap_reduce" if produced is not None else "")
            self._train_launches = 3                     # epoch flag, sample order copy, graph replay
            return last
        ready = ReadySpec(cf_ptr, self.chunk_elems, epoch - 1) if fused else None

        def wait_chunks(rng):
            if epoch <= 1:
                return
            if rng is None:
                self.ext.wait_flags(cf_ptr, self.n_chunks, epoch - 1)
            else:
                self.ext.wait_flags(cf_ptr + 4 * rng[0], rng[1] - rng[0] + 1, epoch - 1)

        if not fused:
            wait_chunks(None)
        before = lw.launches
        if produced is not None:
            self.ext.set_flag(self.epoch_dev.data_ptr(), epoch - 1)      # the reports publish *epoch_dev + 1
        last = lw.fit(flat, xs, self.y, self.cfg, perm, ready, wait_chunks, produced=produced, before_last_backward=overlapped)
        self._last_path = ("layerwise+fused_bcast" if fused else "layerwise") + ("+overlap_reduce" if produced is not None else "")
        self._train_launches = lw.launches - before
        return last

    def _run_twoshot(self, rounds: int, masks: List[int], host_inputs, read_back: bool) -> RoundReport:
        ext, arena, W, P4, r = self.ext, self.arena, self.world, self.P4, self.rank
        dev = self.device
        deadline = self.round_deadline_ms > 0
        if deadline:
            assert self.coord == 0, "the two-shot deadline protocol takes rank 0 as the coordinator"
            decision_ptrs, global_ptrs = arena.peer_ptrs("decision"), arena.peer_ptrs("global")
        use_prev = abs(self.server_lr - 1.0) > 1e-12
        if use_prev and getattr(self, "theta_prev", None) is None:
            # server_lr != 1: theta <- theta + lr_s (sum_k w_k theta_k - theta) needs the model the round started from, and the
            # ranks train IN PLACE on the arena — every rank keeps a copy (one local P-element pass per round)
            self.theta_prev = torch.empty(P4, device=dev)
        work_ptrs = arena.peer_ptrs("work")
        shadow_ptrs = arena.peer_ptrs("shadow") if self.bf16_shadow else []
        cflag_ptrs = arena.peer_ptrs("chunk_flags")
        arrive_ptrs = [arena.ptr("flags", k, 1 + r) for k in range(W)]  # my arrive slot on every rank
        n_blocks = max(1, min(148 * 2, (self.n_chunks + W - 1) // W))
        losses_log = torch.zeros(rounds, W, 2, device=dev)
        launches = 0
        e0 = self.epoch
        if _dist_ready() and W > 1 and self._barrier:
            dist.barrier(group=self.group)
            self._align_streams()
        torch.cuda.synchronize(dev)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        self._phases_begin()
        for i in range(rounds):
            e = e0 + i + 1
            if host_inputs is not None:
                hx, hy = host_inputs[i]
                if self.x is None or self.x.shape != hx.shape:
                    self.x = torch.empty(hx.shape, device=dev, dtype=torch.float32)
                    self.y = torch.empty(hy.shape[0], 1, device=dev)
                    self.set_local_data(self.x, self.y)
                with self._phase("h2d"):
                    self.x.copy_(hx, non_blocking=True)
                    self.y.copy_(hy.view(-1, 1), non_blocking=True)
            wts = self._round_weights(masks[i])
            self.weights_dev[:W].copy_(torch.tensor(wts, dtype=torch.float32), non_blocking=True)
            if use_prev:
                if e > 1:
                    ext.wait_flags(arena.ptr("chunk_flags"), self.n_chunks, e - 1)      # the arena holds the whole previous result
                self.theta_prev.copy_(arena.tensor("work"))
            need_wait = read_back or i == rounds - 1   # otherwise the next round's consumer polls the flags
            sel_w = [w for k, w in enumerate(wts) if (masks[i] >> k) & 1]
            full = (1 << W) - 1
            # NVLS (multimem.ld_reduce sums every member of the multicast group with equal weight inside the switch):
            #   uniform weights over all ranks   -> reduce as is, scale the sum by 1/W in the kernel
            #   n_k weights and / or a subset    -> every rank first scales its own arena by its weight (0 when it was not
            #                                       selected: it presents zeros), the kernel sums with weight 1 over ALL ranks
            nvls = self.use_nvls and arena.has_multicast and W > 1 and not use_prev and bool(sel_w)
            prescale = nvls and (masks[i] != full or max(sel_w) - min(sel_w) >= 1e-7)
            if deadline and prescale:          # (a dropped rank's pre-scaled arena could not be renormalised away inside the switch)
                nvls = prescale = False
            if deadline and e > 1:
                # a rank that missed round e-1's deadline restores its arena from the second arena before it trains again
                ext.wait_flags(arena.ptr("chunk_flags"), self.n_chunks, e - 1)
                ext.twoshot_resync(arena.ptr("decision"), e - 1, r, arena.ptr("work"), arena.ptr("shadow") if self.bf16_shadow else 0,
                                   arena.ptr("global"), P4, 148)
            if prescale:
                self.weights_dev[:W].fill_(1.0)

            def twoshot(blocks: int, produced_ptr: int):
                if deadline:
                    ext.twoshot_fedavg_deadline(work_ptrs, shadow_ptrs, cflag_ptrs, arena.ptr("flags", None, 1), self.weights_dev.data_ptr(),
                                                self.theta_prev.data_ptr() if use_prev else 0, e, masks[i], self.server_lr, P4,
                                                self.chunk_elems, r, blocks, arrive_ptrs, need_wait,
                                                arena.mc_ptr("work") if nvls else 0,
                                                arena.mc_ptr("shadow") if (nvls and self.bf16_shadow) else 0,
                                                self.round_deadline_ms, decision_ptrs, global_ptrs)
                    return
                ext.twoshot_fedavg(work_ptrs, shadow_ptrs, cflag_ptrs, arena.ptr("flags", None, 1), self.weights_dev.data_ptr(),
                                   self.theta_prev.data_ptr() if use_prev else 0, e, full if prescale else masks[i], self.server_lr, P4,
                                   self.chunk_elems, r, blocks,
                                   arrive_ptrs if not produced_ptr else [], need_wait,
                                   arena.mc_ptr("work") if nvls else 0,
                                   arena.mc_ptr("shadow") if (nvls and self.bf16_shadow) else 0,
                                   produced_ptr, self.overlap_timeout_s if produced_ptr else 0.0)

            # fused wgrad -> FedAvg reduce: every rank trains this round, so every rank's last backward reports its chunks
            prod = self._produced_spec() if (masks[i] == full and not prescale and not deadline) else None
            launched = [False]

            def overlapped():
                main = torch.cuda.current_stream(dev)
                self.comm_stream.wait_stream(main)          # weights, epoch flag and the steps before the last backward
                with torch.cuda.stream(self.comm_stream):
                    twoshot(self.overlap_ctas, arena.ptr("produced"))
                launched[0] = True

            if (masks[i] >> r) & 1:
                self._train_launches = 0
                with self._phase("local_fit(+fused_bcast_consume)"):
                    last = self._local_train_inplace(self.rounds_done + i, e, prod, overlapped if prod is not None else None)
                losses_log[i, r, 0] = last
                losses_log[i, r, 1] = last
                launches += self._train_launches
            elif e > 1:
                ext.wait_flags(arena.ptr("chunk_flags"), self.n_chunks, e - 1)
            if launched[0]:
                torch.cuda.current_stream(dev).wait_stream(self.comm_stream)
            else:
                with self._phase("twoshot_reduce_apply_bcast"):
                    if prescale:
                        ext.scale_inplace(arena.ptr("work"), P4, float(wts[r]))
                        launches += 1
                    twoshot(n_blocks, 0)
            self._last_nvls = bool(nvls)
            launches += 1
            if read_back:
                self.loss_host[:2].copy_(losses_log[i, r], non_blocking=True)
                torch.cuda.current_stream(dev).synchronize()
        ev1.record()
        torch.cuda.synchronize(dev)
        phases = self._phases_end()
        self.epoch = e0 + rounds
        self.rounds_done += rounds
        if _dist_ready() and W > 1 and self._barrier:
            dist.barrier(group=self.group)
        nsel = [bin(m).count("1") for m in masks]
        arrived = None
        if deadline:
            ring = arena.tensor("decision").cpu().tolist()
            arrived = [(ring[2 * ((e0 + i + 1) & 7) + 1] if ring[2 * ((e0 + i + 1) & 7)] == e0 + i + 1 else None) for i in range(rounds)]
        self._arrived_masks = arrived
        return RoundReport(rounds, W, "fused", "twoshot", ev0.elapsed_time(ev1), losses_log, launches,
                           bytes_bcast=4 * self.P * sum(nsel), bytes_reduce=4 * self.P * sum(nsel),
                           extra={"provider": arena.provider, "train_path": getattr(self, "_last_path", None), "phases_ms": phases,
                                  "n_chunks": self.n_chunks, "nvls": getattr(self, "_last_nvls", False),
                                  "arrived_masks": getattr(self, "_arrived_masks", None)})

    # ------------------------------------------------------------------------------------------ cpu / gloo
    def _run_cpu(self, rounds: int, masks: List[int]) -> RoundReport:
        W, r = self.world, self.rank
        t0 = time.perf_counter()
        losses_log = torch.zeros(rounds, W, 2)
        self._phases_begin()
        for i in range(rounds):
            with self._phase("bcast"):
                if _dist_ready() and W > 1:
                    dist.broadcast(self.theta, src=self.coord, group=self.group)          # K1
            local = self.theta.clone()
            loss = torch.zeros(())
            if (masks[i] >> r) & 1:
                with self._phase("local_fit"):
                    loss, _ = local_fit(local, self.model, self.x, self.y, self.cfg, self.rounds_done + i)
            w = self._round_weights(masks[i])[r]
            contrib = local * w
            lvec = torch.zeros(W, 2)
            lvec[r, 0] = float(loss)
            with self._phase("reduce_apply"):
                if _dist_ready() and W > 1:
                    dist.reduce(contrib, dst=self.coord, group=self.group)                 # K2 + K3
                    dist.reduce(lvec, dst=self.coord, group=self.group)
                if r == self.coord:
                    self.theta.add_(self.server_lr * (contrib - self.theta))
                    losses_log[i] = lvec
        self.rounds_done += rounds
        nsel = [bin(m).count("1") for m in masks]
        return RoundReport(rounds, W, "cpu", "gloo", (time.perf_counter() - t0) * 1e3, losses_log, 0,
                           bytes_bcast=4 * self.P * sum(nsel), bytes_reduce=4 * self.P * sum(nsel),
                           extra={"phases_ms": self._phases_end()})

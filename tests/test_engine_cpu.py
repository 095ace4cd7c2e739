"""FederatedEngine semantics on CPU: single process and 2 processes over gloo (the host-side logic of
the multi-GPU path), plus the box-mode control plane."""
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from colearn_federated_learning_b200.data import synthetic_unsw
from colearn_federated_learning_b200.models import MLP, flatten_params
from colearn_federated_learning_b200.parallel import FederatedEngine
from colearn_federated_learning_b200.parallel.box import (BoxAgent, BoxControl, DictStore, StoreRelay, parse_box_script, rank_identity,
                                                          worker_id_to_rank)
from colearn_federated_learning_b200.control.event_parser import format_event


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_single_process_round_equals_local_fit_and_loss_decreases(tmp_path):
    eng = FederatedEngine("mlp", backend="cpu", device=torch.device("cpu"), batch_size=4, lr=0.05, seed=3)
    x, y = synthetic_unsw(128, seed=0)
    eng.set_local_data(x, y)
    theta0 = eng.global_flat().clone()
    rep = eng.run_rounds(1)
    assert rep.world == 1 and not torch.equal(eng.global_flat(), theta0)
    first = float(rep.losses[0, 0, 0])
    rep = eng.run_rounds(6)
    assert float(rep.losses[-1, 0, 0]) < first
    path = eng.save_checkpoint(str(tmp_path / "test.pth"))
    m = MLP()
    m.load_state_dict(torch.load(path, weights_only=True))
    assert torch.allclose(flatten_params(m), eng.global_flat())


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        eng = FederatedEngine("mlp", backend="cpu", device=torch.device("cpu"), batch_size=2, lr=0.05, seed=5, weighted=True)
        x, y = synthetic_unsw(90, seed=1)
        lo, hi = [(0, 60), (60, 90)][rank]                      # unequal shards → weighted FedAvg matters
        eng.set_local_data(x[lo:hi], y[lo:hi])
        theta0 = eng.global_flat().clone()
        eng.run_rounds(1)
        # round 2: only rank 1 selected
        eng.run_rounds(1, masks=0b10)
        if rank == 0:
            torch.save({"theta0": theta0, "theta": eng.global_flat().clone(), "counts": eng.counts}, out)
    finally:
        dist.destroy_process_group()


def test_two_process_gloo_weighted_fedavg_and_selection(tmp_path):
    out = str(tmp_path / "res.pt")
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    res = torch.load(out, weights_only=False)
    assert res["counts"] == [60, 30]
    # recompute: both ranks start from theta0; weighted mean 2/3, 1/3; then only rank 1 trains
    x, y = synthetic_unsw(90, seed=1)
    eng = FederatedEngine("mlp", backend="cpu", device=torch.device("cpu"), batch_size=2, lr=0.05, seed=5)
    from colearn_federated_learning_b200.fl.trainer import local_fit
    a, b = res["theta0"].clone(), res["theta0"].clone()
    local_fit(a, eng.model, x[:60], y[:60], eng.cfg, 0)
    local_fit(b, eng.model, x[60:], y[60:], eng.cfg, 0)
    theta1 = (2 / 3) * a + (1 / 3) * b
    c = theta1.clone()
    local_fit(c, eng.model, x[60:], y[60:], eng.cfg, 1)
    assert torch.allclose(res["theta"], c, atol=1e-5)


def _serve_commands(relay, control, executed, stop):
    """What rank 0's main thread does in BoxService.serve: take commands in order, "execute" them, report completion."""
    import json
    while True:
        item = relay.wait_next("commands", stop=stop.is_set)
        if item is None:
            return
        seq, raw = item
        cmd = json.loads(raw)
        executed.append(cmd)
        control.command_done(seq)


def test_store_relay_poll_does_not_wait_for_an_entry_still_being_written():
    """A poll that finds a sequence number taken but its entry not yet set returns what precedes it instead of waiting in the
    store: a c10d store client holds its lock during such a wait, so a writer thread of the same process could not set it."""
    import datetime
    import time
    store = dist.TCPStore("127.0.0.1", 0, 1, True, timeout=datetime.timedelta(seconds=3))
    writer, reader = StoreRelay(store), StoreRelay(store)
    writer.post("events", "first")
    store.add("colearn/box/events/n", 1)                # a second writer has taken number 2 and not set it yet
    t0 = time.time()
    assert reader.poll("events") == ["first"] and time.time() - t0 < 1.0
    store.set("colearn/box/events/2", "second")
    writer.post("events", "third")
    assert reader.poll("events") == ["second", "third"] and reader.poll("events") == []


def test_box_control_plane_builds_selection_mask():
    """Store log -> in-process bus -> parser / registry / temporal window / selection -> `train` command with the mask."""
    import threading
    from colearn_federated_learning_b200.control.window import FakeClock
    store, clock = DictStore(), FakeClock()
    control = BoxControl(StoreRelay(store), 8, 1.0, "topic/state", select_k=4, selection="first", timer_factory=clock, rounds=3)
    executed, stop = [], threading.Event()
    t = threading.Thread(target=_serve_commands, args=(StoreRelay(store), control, executed, stop), daemon=True)
    t.start()
    try:
        agents = [BoxAgent(StoreRelay(store), r, reannounce=False) for r in range(8)]
        for a in agents:
            a.start()
        StoreRelay(store).post("events", "(bad, 1, TRAINING)")                # malformed: ignored
        StoreRelay(store).post("events", "(10.0.0.99, 9999, TRAINING)")        # not a rank of this box: ignored
        assert control.pump() == 10 and len(control.registry) == 8
        clock.advance(1.0)                                                     # window closes: BASELINE config 3 = 4 of 8
        assert executed[0]["op"] == "train" and executed[0]["mask"] == 0b1111 and executed[0]["rounds"] == 3
        assert len(control.history[0]["members"]) == 8 and len(control.registry) == 4   # the unselected four stay registered ...
        clock.advance(1.0)                                                     # ... and the re-armed window trains them next
        assert executed[1]["mask"] == 0b11110000 and len(control.registry) == 0
        # NOT_READY inside the window withdraws a device; a late TRAINING during a training rides the next window
        agents[0].publish("TRAINING"); agents[1].publish("TRAINING"); agents[1].publish("NOT_READY")
        control.pump()
        clock.advance(1.0)
        assert executed[2]["mask"] == 0b1
        # INFERENCE becomes a command for that rank right away
        agents[5].publish("INFERENCE")
        control.pump()
        import time
        deadline = time.time() + 5
        while len(executed) < 4 and time.time() < deadline:                    # taken by the consumer thread
            time.sleep(0.005)
        assert executed[3] == {"op": "inference", "rank": 5, "worker": "10.0.0.6:8782"}
    finally:
        stop.set()
        control.stop()
        t.join(timeout=2)
    assert worker_id_to_rank("10.0.0.6:8782") == 5
    assert parse_box_script("3:NOT_READY:0, 2:inference:1,3:TRAINING:2", 3) == [("NOT_READY", 0), ("TRAINING", 2)]

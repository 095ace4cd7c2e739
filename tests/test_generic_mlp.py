"""The persistent local-SGD kernel for any small MLP (csrc/mlp_generic.cu): one client = one thread-block cluster that splits the
weights, activations all-gathered and backward partials reduced through st.async + mbarrier exchanges.

CPU cases run the kernel source itself through the SIMT shim (csrc/host_shim.h: the CTAs of a cluster run concurrently as OS
threads) and compare it with ``ops.reference``; GPU cases run it on the device and through every caller that picks it
(local_fit, the engine's star round, VirtualWorker training)."""
import os
import re
import shutil
import socket
import subprocess

import pytest
import torch

from colearn_federated_learning_b200 import ops
from colearn_federated_learning_b200.ops import reference

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOSS_CODES = {"bce": 0, "sse": 1, "xent": 2, "mse": 3}
NET = (784, 128, 64, 10)
FFNN = (10, 50, 30, 10, 1)


def _data(dims, loss, n, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(n, dims[0], generator=g)
    y = (torch.randint(0, dims[-1], (n, 1), generator=g).float() if loss == "xent"
         else (torch.rand(n, dims[-1], generator=g) > 0.5).float())
    return x, y


def _theta(dims, seed):
    g = torch.Generator().manual_seed(seed)
    parts = []
    for k, n in zip(dims[:-1], dims[1:]):
        parts += [(torch.rand(n * k, generator=g) * 2 - 1) / k ** 0.5, (torch.rand(n, generator=g) * 2 - 1) / k ** 0.5]
    return torch.cat(parts)


def _ref_fit(theta, dims, act, loss, x, y, perm, batch, lr, epochs, max_steps=-1):
    out = theta.clone()
    last = reference.mlp_local_sgd(out, dims, x, y, perm, batch, lr, epochs, max_steps, loss, act)
    return out, float(last)


# ---------------------------------------------------------------------------------------------------------------- CPU (SIMT)
@pytest.fixture(scope="module")
def simt():
    from colearn_federated_learning_b200.ops import conv
    if shutil.which("g++") is None or not os.path.exists(os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include", "cuda_runtime.h")):
        pytest.skip("no g++ / CUDA headers on this box: the SIMT emulator cannot be built")
    return conv.load_simt()


def _simt_fit(simt, dims, act, loss, theta, xs, ys, perms, batch, lr, epochs, cluster, max_steps=-1, out_scales=None,
              delta=False, flags=None, perm_seed=0, perm_row0=0):
    """K clients in one emulated launch; returns (theta_out per client, losses [K, 2])."""
    K = len(xs)
    outs = [torch.zeros_like(theta) for _ in range(K)]
    losses = torch.zeros(K, 2)
    blob = b""
    for i in range(K):
        perm = perms[i]
        blob += simt.make_client_desc(xs[i].data_ptr(), ys[i].data_ptr(), perm.data_ptr() if perm is not None else 0, theta.data_ptr(),
                                      outs[i].data_ptr(), losses[i].data_ptr(), 0, 0, flags[i:].data_ptr() if flags is not None else 0,
                                      11 + i, xs[i].shape[0], perm.shape[0] if perm is not None else 1, ys[i].shape[1],
                                      1.0 if out_scales is None else out_scales[i], int(delta),
                                      perm_seed if perm is None else 0, perm_row0, 0)
    descs = torch.frombuffer(bytearray(blob), dtype=torch.uint8)
    simt.mlp_local_sgd_generic(list(dims), act == "sigmoid", descs, 0, K, batch, epochs, max_steps, LOSS_CODES[loss], lr, cluster)
    return outs, losses


CPU_CASES = [
    ((12, 40, 24, 3), "none", "xent", 1, 1), ((12, 40, 24, 3), "none", "xent", 2, 1), ((12, 40, 24, 3), "none", "xent", 4, 1),
    ((12, 40, 24, 3), "none", "xent", 2, 3), ((12, 40, 24, 3), "none", "xent", 4, 8),
    ((10, 52, 30, 10, 1), "sigmoid", "bce", 2, 1), ((10, 52, 30, 10, 1), "sigmoid", "bce", 4, 3),
    ((12, 130, 3), "none", "sse", 2, 1), ((12, 130, 3), "none", "mse", 4, 3), ((12, 130, 3), "none", "mse", 1, 8),
]


@pytest.mark.parametrize("dims,act,loss,cluster,batch", CPU_CASES)
def test_generic_kernel_source_on_cpu_matches_reference(simt, dims, act, loss, cluster, batch):
    n, epochs, lr = 29, 2, 0.05                        # 29: a ragged last batch at batch 3 and 8
    x, y = _data(dims, loss, n, seed=len(dims) + batch)
    theta = _theta(dims, seed=cluster)
    perm = reference.make_permutation(n, epochs, seed=5)
    want, last = _ref_fit(theta, dims, act, loss, x, y, perm, batch, lr, epochs)
    (got,), losses = _simt_fit(simt, dims, act, loss, theta, [x], [y], [perm], batch, lr, epochs, cluster)
    torch.testing.assert_close(got, want, rtol=2e-3, atol=2e-4)
    assert abs(float(losses[0, 0]) - last) < 2e-3 * max(1.0, abs(last))


def test_generic_max_steps_cap_on_cpu(simt):
    dims, n, epochs = (12, 40, 24, 3), 29, 2
    x, y = _data(dims, "xent", n, seed=3)
    theta = _theta(dims, seed=3)
    perm = reference.make_permutation(n, epochs, seed=6)
    want, last = _ref_fit(theta, dims, "none", "xent", x, y, perm, 3, 0.05, epochs, max_steps=7)
    (got,), losses = _simt_fit(simt, dims, "none", "xent", theta, [x], [y], [perm], 3, 0.05, epochs, 2, max_steps=7)
    torch.testing.assert_close(got, want, rtol=2e-3, atol=2e-4)
    assert abs(float(losses[0, 0]) - last) < 2e-3 * max(1.0, abs(last))


def test_generic_in_kernel_shuffle_equals_perm_table_on_cpu(simt):
    """perm_seed: the gather computes feistel_index itself — the same order feistel_perm_kernel tabulates, bit for bit."""
    dims, n, epochs, seed, row0 = (12, 40, 24, 3), 37, 2, 987654321, 5
    x, y = _data(dims, "xent", n, seed=8)
    theta = _theta(dims, seed=8)
    table = simt.feistel_permutation(n, row0 + epochs, seed)[row0:].contiguous()
    (a,), la = _simt_fit(simt, dims, "none", "xent", theta, [x], [y], [table], 1, 0.05, epochs, 2)
    (b,), lb = _simt_fit(simt, dims, "none", "xent", theta, [x], [y], [None], 1, 0.05, epochs, 2, perm_seed=seed, perm_row0=row0)
    assert torch.equal(a, b) and torch.equal(la, lb)


def test_generic_several_clients_scale_delta_and_flags_on_cpu(simt):
    dims, n, epochs = (10, 52, 30, 10, 1), 21, 2
    theta = _theta(dims, seed=4)
    xs, ys, perms = [], [], []
    for i in range(3):
        x, y = _data(dims, "bce", n - 4 * i, seed=20 + i)
        xs.append(x)
        ys.append(y)
        perms.append(reference.make_permutation(n - 4 * i, epochs, seed=30 + i))
    scales = [0.5, 0.25, 0.25]
    flags = torch.zeros(3, dtype=torch.int32)
    outs, losses = _simt_fit(simt, dims, "sigmoid", "bce", theta, xs, ys, perms, 1, 0.05, epochs, 2, out_scales=scales, flags=flags)
    douts, _ = _simt_fit(simt, dims, "sigmoid", "bce", theta, xs, ys, perms, 1, 0.05, epochs, 2, out_scales=scales, delta=True)
    for i in range(3):
        want, last = _ref_fit(theta, dims, "sigmoid", "bce", xs[i], ys[i], perms[i], 1, 0.05, epochs)
        torch.testing.assert_close(outs[i], scales[i] * want, rtol=2e-3, atol=2e-4)
        torch.testing.assert_close(douts[i], scales[i] * (want - theta), rtol=2e-3, atol=2e-4)
        assert abs(float(losses[i, 0]) - last) < 2e-3 * max(1.0, abs(last))
    assert flags.tolist() == [11, 12, 13]              # signal_value of client i (raised after its slices landed)


def test_generic_bitwise_reproducible_on_cpu(simt):
    dims, n = (12, 130, 3), 24
    x, y = _data(dims, "mse", n, seed=11)
    theta = _theta(dims, seed=11)
    perm = reference.make_permutation(n, 2, seed=12)
    (a,), la = _simt_fit(simt, dims, "none", "mse", theta, [x], [y], [perm], 3, 0.05, 2, 4)
    (b,), lb = _simt_fit(simt, dims, "none", "mse", theta, [x], [y], [perm], 3, 0.05, 2, 4)
    assert torch.equal(a, b) and torch.equal(la, lb)


def test_generic_plan_rejects_what_the_kernel_cannot_train():
    if not ops._ext.available():
        pytest.skip("CUDA extension not built")
    assert ops.generic_plan((12, 40, 33), "none", 1) is None              # head wider than one warp
    assert ops.generic_plan((8,) * 10, "none", 1) is None                 # 9 layers
    assert ops.generic_plan((784, 1024, 1024, 10), "none", 1) is None     # over the shared memory of 8 CTAs
    assert ops.generic_plan((10, 96, 48, 1), "none", 1, loss="bce") is None   # bce needs a sigmoid head
    assert ops.generic_plan(NET, "none", 1) == 4 and ops.generic_plan(NET, "none", 8) == 8
    assert ops.generic_plan(NET, "none", 1, cluster=2) is None and ops.generic_plan(NET, "none", 1, cluster=8) == 8
    assert ops.generic_plan((10, 96, 48, 1), "sigmoid", 1, loss="bce") == 1
    assert ops.GENERIC_MAX_BATCH <= 8


def test_generic_kernel_sass_exchanges_without_per_step_cluster_barriers():
    """st.async -> STAS, mbarrier try_wait -> SYNCS.PHASECHK.TRANS64.TRYWAIT; barrier.cluster (UCGABAR_ARV) only in the
    prologue and the epilogue; no spills (-Xptxas -v).  Cross-compiled: no GPU needed."""
    nvcc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    if not os.path.exists(nvcc) or shutil.which("cuobjdump") is None:
        pytest.skip("needs nvcc and cuobjdump")
    from colearn_federated_learning_b200.ops import build
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        obj = os.path.join(tmp, "g.o")
        cc = subprocess.run([nvcc, *build.NVCC_FLAGS, "-I", build.CSRC, "-c", os.path.join(build.CSRC, "mlp_generic.cu"), "-o", obj],
                            capture_output=True, text=True, timeout=600)
        assert cc.returncode == 0, cc.stdout + cc.stderr
        sass = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, timeout=300).stdout
    log = cc.stdout + cc.stderr
    spills = re.findall(r"Compiling entry function '(\S*mlp_local_sgd_generic_kernel\S*)'.*?(\d+) bytes spill stores", log, re.S)
    assert spills and all(int(s) == 0 for _, s in spills), log
    body = sass[sass.index("mlp_local_sgd_generic_kernel"):]
    assert "STAS" in body and "SYNCS.PHASECHK.TRANS64.TRYWAIT" in body
    assert body.count("UCGABAR_ARV") == 2, body.count("UCGABAR_ARV")


# ------------------------------------------------------------------------------------------------------------------------ GPU
def _gpu_fit(dims, act, loss, theta, x, y, perm, batch, lr, epochs, cluster):
    """One client through the generic kernel itself (also for dims that have a specialised kernel)."""
    dev = torch.device("cuda", 0)
    out = theta.to(dev).clone()
    loss_out = torch.zeros(2, device=dev)
    task = ops.ClientTask(x=x.to(dev).contiguous(), y=y.to(dev).contiguous(), theta_in=out, theta_out=out,
                          perm=perm.to(dev, torch.int32).contiguous(), loss_out=loss_out)
    descs = ops.build_client_descs([task], dev)
    ops._ext.require().mlp_local_sgd_generic(list(dims), act == "sigmoid", descs, 0, 1, batch, epochs, -1, LOSS_CODES[loss], lr, cluster)
    torch.cuda.synchronize()
    return out.cpu(), loss_out.cpu()


GPU_MODELS = [
    (NET, "none", "xent", 1), (NET, "none", "xent", 8), ((10, 96, 48, 1), "sigmoid", "bce", 1), ((2, 16, 16, 2), "none", "xent", 1),
    ((16, 40, 40, 40, 40, 40, 40, 4), "none", "xent", 3), (FFNN, "sigmoid", "bce", 1), (FFNN, "sigmoid", "sse", 4),
]


@pytest.mark.gpu
@pytest.mark.parametrize("dims,act,loss,batch", GPU_MODELS)
def test_generic_kernel_matches_reference_at_every_legal_cluster(dims, act, loss, batch):
    n, epochs, lr = (96 if dims == NET else 150), 2, 0.02
    x, y = _data(dims, loss, n, seed=len(dims) * 7 + batch)
    theta = _theta(dims, seed=batch)
    perm = reference.make_permutation(n, epochs, seed=9)
    want, last = _ref_fit(theta, dims, act, loss, x, y, perm, batch, lr, epochs)
    legal = [c for c in (1, 2, 4, 8) if ops.generic_plan(dims, act, batch, c, loss) is not None]
    assert legal and (dims != FFNN or 8 in legal)      # C = 8 on the FFNN: 7 CTAs own no head row
    for c in legal:
        got, lo = _gpu_fit(dims, act, loss, theta, x, y, perm, batch, lr, epochs, c)
        torch.testing.assert_close(got, want, rtol=2e-3, atol=2e-4, msg=lambda m: f"cluster {c}: {m}")
        assert abs(float(lo[0]) - last) < 2e-3 * max(1.0, abs(last)), (c, float(lo[0]), last)


@pytest.mark.gpu
def test_generic_kernel_bitwise_reproducible_on_gpu():
    x, y = _data(NET, "xent", 64, seed=1)
    theta = _theta(NET, seed=1)
    perm = reference.make_permutation(64, 1, seed=2)
    a, la = _gpu_fit(NET, "none", "xent", theta, x, y, perm, 1, 0.02, 1, 4)
    b, lb = _gpu_fit(NET, "none", "xent", theta, x, y, perm, 1, 0.02, 1, 4)
    assert torch.equal(a, b) and torch.equal(la, lb)


@pytest.mark.gpu
def test_local_fit_of_net_takes_the_generic_kernel_at_small_batch():
    from colearn_federated_learning_b200.fl import trainer
    from colearn_federated_learning_b200.models import build_model, flatten_params
    torch.manual_seed(0)
    model = build_model("net").cuda()
    x, y = _data(NET, "xent", 128, seed=3)
    flat0 = flatten_params(model).cuda()
    cfg = trainer.FitConfig(model="net", loss="xent", batch_size=1, lr=0.02, shuffle=False)
    flat = flat0.clone()
    _, path = trainer.local_fit(flat, model, x.cuda(), y.cuda(), cfg)
    assert path == "persistent" and trainer.LAST_FIT_LAUNCHES == 1
    want, _ = _ref_fit(flat0.cpu(), NET, "none", "xent", x, y, reference.make_permutation(128, 1, 0, shuffle=False), 1, 0.02, 1)
    torch.testing.assert_close(flat.cpu(), want, rtol=2e-3, atol=2e-4)
    cfg32 = trainer.FitConfig(model="net", loss="xent", batch_size=32, lr=0.02, shuffle=False)
    _, path = trainer.local_fit(flat0.clone(), model, x.cuda(), y.cuda(), cfg32)
    assert path == "layerwise"


def _engine_reference(theta0, x, y, sizes_bounds, rounds, lr):
    ref = theta0.clone()
    n = x.shape[0]
    for _ in range(rounds):
        acc = torch.zeros_like(ref)
        for lo, hi in sizes_bounds:
            loc = ref.clone()
            reference.mlp_local_sgd(loc, NET, x[lo:hi], y[lo:hi], reference.make_permutation(hi - lo, 1, 0, shuffle=False), 1, lr, 1, -1,
                                    "xent")
            acc += loc * ((hi - lo) / n)
        ref = acc
    return ref


@pytest.mark.gpu
@pytest.mark.parametrize("clients", [1, 3])
def test_engine_star_round_for_net(clients):
    from colearn_federated_learning_b200.data import shard_bounds
    from colearn_federated_learning_b200.parallel import FederatedEngine
    dev = torch.device("cuda", 0)
    eng = FederatedEngine("net", backend="fused", device=dev, batch_size=1, lr=0.02, seed=7, shuffle=False, weighted=True,
                          clients_per_rank=clients)
    assert eng.algo == "star"
    n = 90
    x, y = _data(NET, "xent", n, seed=4)
    eng.set_local_data(x, y)
    theta0 = eng.global_flat().cpu().clone()
    rep = eng.run_rounds(2)
    assert rep.algo == "star"
    bounds = [(0, n)] if clients == 1 else list(shard_bounds(n, clients))
    ref = _engine_reference(theta0, x, y, bounds, 2, 0.02)
    assert torch.allclose(eng.global_flat().cpu(), ref, atol=5e-4, rtol=5e-3), (eng.global_flat().cpu() - ref).abs().max()
    assert rep.launches == 2 * (2 if clients == 1 else 3) + 1 and torch.isfinite(rep.losses).all()


@pytest.mark.gpu
def test_virtual_workers_of_net_train_in_one_launch(monkeypatch):
    from colearn_federated_learning_b200.control import coordinator
    from colearn_federated_learning_b200.fl.trainer import FitConfig
    from colearn_federated_learning_b200.models import build_model, flatten_params

    class Shard:
        def __init__(self, x, y):
            self.x, self.y = x, y

        def __len__(self):
            return self.x.shape[0]

    class Fed:
        def __init__(self, shards):
            self.workers = list(range(len(shards)))
            self.shards = shards

        def __getitem__(self, w):
            return self.shards[w]

    dev = torch.device("cuda", 0)
    shards = []
    for i in range(5):
        x, y = _data(NET, "xent", 20 + 3 * i, seed=50 + i)
        shards.append(Shard(x.to(dev), y.to(dev)))
    torch.manual_seed(1)
    model = build_model("net").to(dev)
    theta = flatten_params(model).to(dev)
    cfg = FitConfig(model="net", loss="xent", batch_size=1, lr=0.02, shuffle=False)
    calls = []
    real = ops.mlp_local_sgd_multi
    monkeypatch.setattr(coordinator.ops, "mlp_local_sgd_multi", lambda *a, **k: (calls.append(a[3]), real(*a, **k))[1])
    flats, losses, counts = coordinator.train_virtual_workers(theta, model, Fed(shards), cfg, 0)
    assert calls == [5]                                 # one launch, five clusters
    for i, sh in enumerate(shards):
        want, last = _ref_fit(theta.cpu(), NET, "none", "xent", sh.x.cpu(), sh.y.cpu(),
                              reference.make_permutation(len(sh), 1, 0, shuffle=False), 1, 0.02, 1)
        torch.testing.assert_close(flats[i].cpu(), want, rtol=2e-3, atol=2e-4)
        assert abs(losses[i] - last) < 2e-3 * max(1.0, abs(last))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _star_rank_main(rank, world, port, out_path):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from colearn_federated_learning_b200.parallel import FederatedEngine
        dev = torch.device("cuda", rank)
        sizes = [60, 40]
        x, y = _data(NET, "xent", sizes[rank], seed=70 + rank)
        eng = FederatedEngine("net", backend="fused", device=dev, batch_size=1, lr=0.02, seed=3, shuffle=False, weighted=True)
        eng.set_local_data(x, y)
        theta0 = eng.global_flat().cpu().clone()
        rep = eng.run_rounds(2)
        gathered = [None] * world
        dist.all_gather_object(gathered, (x, y))
        if rank == 0:
            theta = theta0
            for _ in range(2):
                acc = torch.zeros_like(theta)
                for k in range(world):
                    loc = theta.clone()
                    xs, ys = gathered[k]
                    reference.mlp_local_sgd(loc, NET, xs, ys, reference.make_permutation(len(xs), 1, 0, shuffle=False), 1, 0.02, 1, -1, "xent")
                    acc += loc * (sizes[k] / sum(sizes))
                theta = acc
            torch.save({"err": (eng.global_flat().cpu() - theta).abs().max().item(), "algo": rep.algo}, out_path)
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.multigpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_engine_star_round_for_net_on_two_gpus(tmp_path):
    import torch.multiprocessing as mp
    out = str(tmp_path / "out.pt")
    mp.spawn(_star_rank_main, args=(2, _free_port(), out), nprocs=2, join=True)
    res = torch.load(out, weights_only=False)
    assert res["algo"] == "star" and res["err"] < 2e-3, res

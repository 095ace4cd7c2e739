"""Python face of ``mlp_local_sgd_persistent`` (csrc/mlp_persistent.cu) — SURVEY K12.

One launch runs the *entire* local fit of one or many federated clients (one CTA each): the
reference's per-batch ``zero_grad → forward → loss → backward → step`` loop
(``client_federated.py:101-120`` locally; PySyft ``_fit`` remotely, SURVEY C27) never returns to
the host.  Supported architectures are the compile-time instantiations FFNN (10-50-30-10-1,
sigmoid), MLP (10-64-64-2) and TestingRemote (2-50-10-1).  Every other MLP with at most 8 layers and a head of at
most 32 outputs runs the run-time-shaped kernel of ``csrc/mlp_generic.cu`` (one client = one thread-block cluster that
splits the weights); callers prefer it to the layer-wise trainer (``fl/layerwise.py``) up to ``GENERIC_MAX_BATCH``.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Optional, Sequence, Tuple, Union

import torch

from . import _ext, host, reference

NET_KINDS = {
    ((10, 50, 30, 10, 1), "sigmoid"): 0,
    ((10, 64, 64, 2), "none"): 1,
    ((2, 50, 10, 1), "none"): 2,
}
LOSS_CODES = {"bce": 0, "sse": 1, "xent": 2, "mse": 3}
# Kernel variants: 5 = register-resident weights, 128-thread CTA, blocked reduction slices (LDS.128) + pre-scaled dz;
# 6 = 5 with packed fp32 math (fma.rn.f32x2 -> SASS FFMA2); 3 = strided slices (the round-1 default); 1 = smem-resident
# weights (first version).  Measured on a B200 (us per batch-1 SGD step, profiles/README.md R2.9: the head's sigmoid on single
# MUFU instructions, loss value without a divergent branch, narrow heads held whole in every lane, the FFNN's 30 -> 10 layer
# computed per warp):
#                   v1      v3      v5      v6
#   MLP 10-64-64-2  1.646   0.670   0.624   0.579     <- 64-wide layers: every dot product / update is FFMA2-shaped
#   FFNN            1.627   0.668   0.616   0.577     <- (was 0.711 / 0.716 before those four changes)
# 0 (default) picks the fastest measured variant per net.
KERNEL_VARIANT = int(__import__("os").environ.get("COLEARN_MLP_VARIANT", "0"))
BEST_VARIANT = {0: 6, 1: 6, 2: 5}          # net kind (NET_KINDS values) -> variant


def resolve_variant(kind: int, variant: Optional[int] = None) -> int:
    v = KERNEL_VARIANT if variant is None else int(variant)
    return BEST_VARIANT.get(kind, 5) if v == 0 else v


# Largest batch at which the callers (fl/trainer.local_fit, the engine's star round, train_virtual_workers) prefer the generic
# kernel to the layer-wise tcgen05 trainer for an MLP without a specialised kernel.  profiles/README.md R3.1 has the measured
# crossover; the cap stays at 8 so that larger batches keep the layer-wise / two-shot paths they take today.
GENERIC_MAX_BATCH = 8
GENERIC_MAX_LAYERS = 8
GENERIC_MAX_DOUT = 32

PtrLike = Union[torch.Tensor, int, None]


def net_kind_for(dims: Sequence[int], out_activation: str = "none") -> Optional[int]:
    return NET_KINDS.get((tuple(int(d) for d in dims), out_activation))


def generic_plan(dims: Sequence[int], out_activation: str, batch_size: int, cluster: int = 0,
                 loss: Optional[str] = None) -> Optional[int]:
    """Cluster size (CTAs per client) the generic kernel uses for this MLP, or None when it cannot train it: a head wider
    than 32, more than 8 layers, an output activation other than none / sigmoid, ``bce`` without a sigmoid head, or weights
    that do not fit the shared memory of 8 CTAs.  ``cluster`` > 0 asks for that size (None if it is not legal or does not
    fit)."""
    dims = [int(d) for d in dims]
    if len(dims) < 2 or len(dims) - 1 > GENERIC_MAX_LAYERS or dims[-1] > GENERIC_MAX_DOUT or min(dims) < 1:
        return None
    if out_activation not in ("none", "sigmoid") or (loss == "bce" and out_activation != "sigmoid"):
        return None
    c = int(_ext.require().mlp_generic_plan(dims, max(1, int(batch_size)), int(cluster)))
    return c if c > 0 else None


def persistent_path(dims: Sequence[int], out_activation: str, batch_size: int, loss: Optional[str] = None, device=None) -> bool:
    """True when a whole local fit of this MLP is one persistent-kernel launch on ``device``: a specialised kernel
    (NET_KINDS), or — on a CUDA device, up to GENERIC_MAX_BATCH — the generic one."""
    if net_kind_for(dims, out_activation) is not None:
        return True
    if device is not None and torch.device(device).type != "cuda":
        return False
    return int(batch_size) <= GENERIC_MAX_BATCH and generic_plan(dims, out_activation, batch_size, loss=loss) is not None


def _ptr(t: PtrLike) -> int:
    if t is None:
        return 0
    if isinstance(t, torch.Tensor):
        return t.data_ptr()
    return int(t)


@dataclass
class ClientTask:
    """Everything one client CTA needs.  Pointers may be tensors or raw ints (peer memory)."""

    x: torch.Tensor                      # [n, d_in] fp32 CUDA
    y: torch.Tensor                      # [n, y_dim] fp32 CUDA (xent: class index as float)
    theta_in: PtrLike                    # flat arena to start from
    theta_out: PtrLike                   # destination of out_scale * theta_k (or delta)
    perm: Optional[torch.Tensor] = None  # int32 [rows, n]
    loss_out: PtrLike = None             # float[2]: last / mean loss
    wait_flag: PtrLike = None
    wait_value: int = 0
    signal_flag: PtrLike = None
    signal_value: int = 0
    out_scale: float = 1.0
    delta_mode: bool = False
    perm_seed: int = 0                   # != 0 with perm=None: the kernel tabulates the keyed Feistel order itself (before it
    perm_row0: int = 0                   # waits for the broadcast); epoch e = row perm_row0 + e of device_permutation(n, *, perm_seed)
    perm_scratch: Optional[torch.Tensor] = None   # int32 [epochs of the fit * n] device scratch for that table (required with perm_seed)
    _keep: list = field(default_factory=list, repr=False)

    def pack(self) -> bytes:
        ext = _ext.require()
        n = int(self.x.shape[0])
        if self.perm is None and self.perm_seed:
            assert self.perm_scratch is not None and self.perm_scratch.dtype == torch.int32 and self.perm_scratch.numel() >= n, \
                "perm_seed needs an int32 perm_scratch of >= epochs * n elements on the kernel's device"
        y_dim = int(self.y.shape[1]) if self.y.dim() == 2 else 1
        rows = int(self.perm.shape[0]) if self.perm is not None else 1
        return ext.make_client_desc(_ptr(self.x), _ptr(self.y), _ptr(self.perm), _ptr(self.theta_in),
                                    _ptr(self.theta_out), _ptr(self.loss_out), _ptr(self.wait_flag),
                                    int(self.wait_value), _ptr(self.signal_flag), int(self.signal_value),
                                    n, rows, y_dim, float(self.out_scale), int(bool(self.delta_mode)),
                                    int(self.perm_seed) if self.perm is None else 0, int(self.perm_row0), _ptr(self.perm_scratch))


def build_client_descs(tasks: Sequence[ClientTask], device) -> torch.Tensor:
    """Pack descriptors into one uint8 CUDA tensor (pinned staging → async H2D)."""
    blob = b"".join(t.pack() for t in tasks)
    host = torch.frombuffer(bytearray(blob), dtype=torch.uint8)
    if torch.cuda.is_available():
        host = host.pin_memory()
    return host.to(device, non_blocking=True)


def _prep_xy(x: torch.Tensor, y: torch.Tensor, loss: str) -> Tuple[torch.Tensor, torch.Tensor]:
    x = x.contiguous().float()
    y = y.contiguous().float()
    if y.dim() == 1:
        y = y.view(-1, 1)
    return x, y


def mlp_local_sgd_multi(dims: Sequence[int], out_activation: str, descs: torch.Tensor, n_clients: int,
                        batch_size: int = 1, lr: float = 0.01, epochs: int = 1, max_nr_batches: int = -1,
                        loss: str = "xent", desc_offset: int = 0, variant: Optional[int] = None, cluster: int = 0) -> None:
    """Launch ``n_clients`` clients from a packed descriptor tensor (see :func:`build_client_descs`): one CTA each for the
    specialised networks, one cluster each for any other MLP (``cluster`` forces its size; tests)."""
    kind = net_kind_for(dims, out_activation)
    if loss == "bce" and out_activation != "sigmoid":
        raise ValueError("bce needs a sigmoid head")
    if kind is None:
        c = generic_plan(dims, out_activation, batch_size, cluster, loss)
        if c is None:
            raise ValueError(f"no persistent kernel for dims={tuple(dims)} act={out_activation} batch={batch_size} "
                             f"cluster={cluster}: the generic kernel takes <= {GENERIC_MAX_LAYERS} layers, a head of "
                             f"<= {GENERIC_MAX_DOUT} and weights that fit 8 CTAs")
        _ext.require().mlp_local_sgd_generic([int(d) for d in dims], out_activation == "sigmoid", descs, int(desc_offset),
                                             int(n_clients), int(batch_size), int(epochs),
                                             int(max_nr_batches if max_nr_batches is not None else -1), LOSS_CODES[loss],
                                             float(lr), c)
        return
    _ext.require().mlp_local_sgd(kind, descs, int(desc_offset), int(n_clients), int(batch_size), int(epochs),
                                 int(max_nr_batches if max_nr_batches is not None else -1), LOSS_CODES[loss], float(lr),
                                 resolve_variant(kind, variant))


def mlp_local_sgd(flat: torch.Tensor, dims: Sequence[int], x: torch.Tensor, y: torch.Tensor,
                  perm: Optional[torch.Tensor], batch_size: int = 1, lr: float = 0.01, epochs: int = 1,
                  max_nr_batches: int = -1, loss: str = "xent", out_activation: str = "none",
                  return_mean: bool = False, variant: Optional[int] = None, cluster: int = 0) -> torch.Tensor:
    """Single-client in-place local SGD on ``flat``; returns the last batch loss (0-dim tensor).

    CPU tensors run ``reference.mlp_local_sgd`` (identical semantics); CUDA tensors run the
    persistent kernel — there is no silent fallback on CUDA."""
    if not flat.is_cuda:
        # CPU devices: the native host executor (csrc/mlp_host.cpp) when it is built and the arena can be trained in
        # place, else the PyTorch definitions (identical semantics; the executor is tested against them)
        if (host.available() and flat.dtype == torch.float32 and flat.is_contiguous() and not flat.requires_grad
                and out_activation in ("none", "sigmoid")):
            res = host.mlp_local_sgd_multi(dims, out_activation, [flat], [x], [y], [perm], batch_size, lr, epochs,
                                           max_nr_batches, loss, threads=1)
            return res[0, 1 if return_mean else 0].clone()
        if perm is None:
            perm = reference.make_permutation(x.shape[0], epochs, 0, shuffle=False)
        return reference.mlp_local_sgd(flat, dims, x, y, perm, batch_size, lr, epochs, max_nr_batches, loss, out_activation)
    x, y = _prep_xy(x, y, loss)
    loss_out = torch.zeros(2, device=flat.device, dtype=torch.float32)
    if perm is not None:
        perm = perm.to(flat.device, torch.int32).contiguous()
    task = ClientTask(x=x, y=y, theta_in=flat, theta_out=flat, perm=perm, loss_out=loss_out)
    descs = build_client_descs([task], flat.device)
    mlp_local_sgd_multi(dims, out_activation, descs, 1, batch_size, lr, epochs, max_nr_batches, loss, variant=variant,
                        cluster=cluster)
    return loss_out[1 if return_mean else 0]


def mlp_forward(flat: torch.Tensor, dims: Sequence[int], x: torch.Tensor, out_activation: str = "none") -> torch.Tensor:
    """Batched forward of a small MLP from its flat arena (inference / evaluation)."""
    if not flat.is_cuda:
        return reference.mlp_forward(flat, dims, x, out_activation)[0]
    kind = net_kind_for(dims, out_activation)
    if kind is None:
        raise ValueError(f"no persistent-kernel instantiation for dims={tuple(dims)}")
    return _ext.require().mlp_forward(kind, flat.contiguous(), x.contiguous().float(), int(dims[-1]))

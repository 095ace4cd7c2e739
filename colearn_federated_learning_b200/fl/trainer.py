"""Worker-side fit executor.

Re-creates the contract of PySyft's ``FederatedClient.fit/_fit`` (SURVEY C27, [EXTERNAL]) that
the reference triggers with ``worker.async_fit(dataset_key="training")``
(``client_federated.py:210``): build SGD(lr), iterate shuffled batches for ``epochs`` epochs, stop
after ``max_nr_batches`` steps, return the last loss — but on a flat fp32 arena and, for the
small MLP family on a GPU, as ONE persistent-kernel launch (``ops.mlp_local_sgd``).

Three execution paths, chosen by :func:`local_fit`:
  * ``persistent``  FFNN / MLP / TestingRemote on CUDA → csrc/mlp_persistent.cu; any other MLP that fits the generic
                    kernel at batch <= ops.GENERIC_MAX_BATCH → csrc/mlp_generic.cu
  * ``layerwise``   wide MLPs on CUDA → tcgen05 GEMMs + fused loss/SGD kernels (fl/layerwise.py)
  * ``convnet``     ResNet-18 on CUDA → im2col + tcgen05 GEMMs + this repo's BatchNorm / pooling kernels
                    (fl/convnet.py); ``COLEARN_CONV_PATH=torch`` selects the library path instead
  * ``torch``       anything else (every model on CPU; conv nets with a ragged last batch) → autograd loop
                    that still uses this repo's fused loss + flat SGD kernels where they apply.
"""
from __future__ import annotations

import logging
import os
from dataclasses import dataclass, asdict
from typing import Any, Dict, Optional, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import ops
from ..models import MLPNet, flatten_params, unflatten_params, DEFAULT_LOSS
from ..ops import reference


@dataclass
class FitConfig:
    """What the coordinator ships instead of a PySyft ``TrainConfig`` (cf.py:199-208)."""

    model: str = "ffnn"
    loss: str = "bce"
    batch_size: int = 1
    epochs: int = 1
    max_nr_batches: int = -1
    lr: float = 0.01
    shuffle: bool = True
    seed: int = 1
    optimizer: str = "SGD"

    def to_dict(self) -> Dict[str, Any]:
        return asdict(self)

    @classmethod
    def from_dict(cls, d: Dict[str, Any]) -> "FitConfig":
        return cls(**{k: v for k, v in d.items() if k in cls.__dataclass_fields__})


# Which executor trains conv nets on a GPU: "native" = fl/convnet.py (this repo's kernels), "torch" = autograd over
# cuDNN/ATen.  ``COLEARN_CONV_PATH`` overrides; on CPU tensors the native path (PyTorch definitions of the same ops)
# only runs when asked for explicitly.
CONV_PATH_DEFAULT = "native"

# kernels of THIS repo launched by the most recent local_fit (library kernels of the torch path are not counted);
# the engine adds it to RoundReport.launches
LAST_FIT_LAUNCHES = 0


def conv_path(device) -> str:
    env = os.environ.get("COLEARN_CONV_PATH", "").strip().lower()
    if env in ("native", "torch"):
        return env
    return CONV_PATH_DEFAULT if torch.device(device).type == "cuda" else "torch"


def resolve_loss(model_name: str, loss: str) -> str:
    return DEFAULT_LOSS.get(model_name, "xent") if loss in ("auto", None, "") else loss


def make_perm(n: int, cfg: FitConfig, device, round_idx: int = 0) -> Optional[torch.Tensor]:
    if not cfg.shuffle:
        return None
    seed = cfg.seed * 7919 + round_idx
    if torch.device(device).type == "cuda":
        return ops.device_permutation(n, cfg.epochs, seed, device)
    return reference.make_permutation(n, cfg.epochs, seed)


def _loss_torch(out: torch.Tensor, y: torch.Tensor, loss: str) -> torch.Tensor:
    if loss == "xent":
        return F.cross_entropy(out.float(), y.reshape(-1).long())
    y = y.reshape(out.shape).to(out.dtype)
    if loss == "bce":
        return F.binary_cross_entropy(out, y)
    if loss == "sse":
        return ((out - y) ** 2).sum()
    if loss == "mse":
        return ((out - y) ** 2).sum() / out.shape[0]
    raise ValueError(loss)


def torch_fit(model: nn.Module, x: torch.Tensor, y: torch.Tensor, cfg: FitConfig, perm: Optional[torch.Tensor],
              autocast_bf16: bool = False) -> torch.Tensor:
    """Generic autograd fit (library conv/BN kernels) with a flat in-place SGD step."""
    model.train()
    params = [p for p in model.parameters()]
    n = x.shape[0]
    it = 0
    limit = cfg.max_nr_batches if cfg.max_nr_batches and cfg.max_nr_batches > 0 else None
    last = torch.zeros((), device=x.device)
    for e in range(cfg.epochs):
        order = perm[e % perm.shape[0]].long() if perm is not None else torch.arange(n, device=x.device)
        for lo in range(0, n, cfg.batch_size):
            idx = order[lo:lo + cfg.batch_size]
            for p in params:
                p.grad = None
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast_bf16 and x.is_cuda):
                out = model(x[idx])
            last = _loss_torch(out, y[idx], cfg.loss)
            last.backward()
            with torch.no_grad():
                for p in params:
                    if p.grad is not None:
                        if p.is_cuda and p.dtype == torch.float32 and p.is_contiguous() and p.grad.is_contiguous():
                            ops.sgd_step(p.data.view(-1), p.grad.view(-1), cfg.lr)
                        else:
                            p.sub_(p.grad, alpha=cfg.lr)
            it += 1
            if limit is not None and it >= limit:
                return last.detach()
    return last.detach()


def local_fit(flat: torch.Tensor, model: nn.Module, x: torch.Tensor, y: torch.Tensor, cfg: FitConfig,
              round_idx: int = 0, perm: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, str]:
    """Run the local fit **in place on ``flat``**; returns (last loss, path used)."""
    global LAST_FIT_LAUNCHES
    LAST_FIT_LAUNCHES = 0
    loss = resolve_loss(cfg.model, cfg.loss)
    cfg = FitConfig(**{**cfg.to_dict(), "loss": loss})
    if perm is None:
        perm = make_perm(x.shape[0], cfg, flat.device, round_idx)
    if isinstance(model, MLPNet):
        spec = model.spec
        xx = x.view(x.shape[0], -1) if spec.flatten_input else x
        has_kernel = ops.persistent_path(spec.dims, spec.out_activation, cfg.batch_size, loss, flat.device)
        if not flat.is_cuda or has_kernel:
            last = ops.mlp_local_sgd(flat, spec.dims, xx, y, perm, cfg.batch_size, cfg.lr, cfg.epochs,
                                     cfg.max_nr_batches, loss, spec.out_activation)
            LAST_FIT_LAUNCHES = 1 if flat.is_cuda else 0
            return last, ("persistent" if flat.is_cuda else "reference")
        if flat.is_cuda:
            from .layerwise import LayerwiseMLPTrainer
            if LayerwiseMLPTrainer.supports(spec, cfg):
                tr = LayerwiseMLPTrainer.cached(spec, flat, cfg.batch_size)
                before = tr.launches
                last = tr.fit(flat, xx, y, cfg, perm)
                LAST_FIT_LAUNCHES = tr.launches - before
                return last, "layerwise"
    if conv_path(flat.device) == "native":
        from .convnet import ConvNetTrainer
        if ConvNetTrainer.supports(model, cfg, x):
            tr = ConvNetTrainer.cached(model, flat, cfg.batch_size, tuple(x.shape[2:]))
            before = tr.launches
            last = tr.fit(flat, model, x, y, cfg, perm)
            LAST_FIT_LAUNCHES = tr.launches - before
            return last, "convnet"
    if flat.is_cuda:
        _library_path_guard(model, cfg, x)
    unflatten_params(model, flat)
    last = torch_fit(model, x, y, cfg, perm, autocast_bf16=flat.is_cuda)
    flatten_params(model, out=flat)
    return last, "torch"


_WARNED_LIBRARY_PATH: set = set()


def _library_path_guard(model: nn.Module, cfg: FitConfig, x: torch.Tensor) -> None:
    """CUDA tensors never reach autograd + cuBLAS / cuDNN silently (DESIGN.md §3).

    * The architectures this repo ships kernels for — every :class:`MLPNet` and ``ResNet18`` — must train on them: a shape
      the kernels do not cover (e.g. a ResNet shard that is not a whole number of 128-image batches, or images smaller
      than 32x32) RAISES here instead of quietly switching libraries.  ``COLEARN_CONV_PATH=torch`` is the explicit request
      for the cuDNN path of conv nets, ``COLEARN_ALLOW_AUTOGRAD=1`` the general one.
    * A user-registered architecture (``models.register_model`` with an arbitrary ``nn.Module``) has no hand-written
      kernels by construction; it trains through autograd with this repo's flat SGD step, announced once per class."""
    from ..models.resnet import ResNet18
    allow = os.environ.get("COLEARN_ALLOW_AUTOGRAD", "0") == "1"
    builtin = isinstance(model, (MLPNet, ResNet18))
    explicit_conv = isinstance(model, ResNet18) and os.environ.get("COLEARN_CONV_PATH", "").strip().lower() == "torch"
    if builtin and not (allow or explicit_conv):
        what = (f"MLP {tuple(model.spec.dims)} with loss={cfg.loss!r}, batch_size={cfg.batch_size}" if isinstance(model, MLPNet) else
                f"ResNet18 on input {tuple(x.shape)} with loss={cfg.loss!r}, batch_size={cfg.batch_size} "
                "(the conv kernels need xent, batch_size % 128 == 0, shard size % batch_size == 0, images >= 32x32)")
        raise RuntimeError(f"no sm_100a kernel path for {what}; refusing to fall back to autograd + cuBLAS/cuDNN on a CUDA tensor. "
                           "Set COLEARN_ALLOW_AUTOGRAD=1 (or COLEARN_CONV_PATH=torch for conv nets) to request the library path.")
    key = type(model).__name__
    if key not in _WARNED_LIBRARY_PATH:
        _WARNED_LIBRARY_PATH.add(key)
        logging.getLogger(__name__).warning("%s trains through autograd + library kernels (%s); only this repo's flat SGD step is its own",
                                            key, "requested by environment" if (allow or explicit_conv) else "user-registered architecture")

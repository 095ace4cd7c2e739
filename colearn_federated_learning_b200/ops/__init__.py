"""Hot ops.  CUDA tensors → hand-written sm_100a kernels (``csrc/``); CPU tensors → ``reference``.

There is deliberately no silent GPU fallback: a CUDA tensor with the extension missing raises.
"""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import torch

from . import reference
from . import _ext
from . import host  # noqa: F401  (native CPU executor of the MLP local fit)
from .fused_mlp import (NET_KINDS, LOSS_CODES, net_kind_for, mlp_local_sgd, mlp_local_sgd_multi,  # noqa: F401
                        mlp_forward, ClientTask, build_client_descs, generic_plan, persistent_path, GENERIC_MAX_BATCH)
from .reference import make_permutation, total_steps  # noqa: F401


def _cuda(t: torch.Tensor) -> bool:
    return t.is_cuda


def sgd_step(param: torch.Tensor, grad: torch.Tensor, lr: float) -> torch.Tensor:
    """``param -= lr * grad`` in place on a flat fp32 arena (SURVEY K12)."""
    if _cuda(param):
        _ext.require().sgd_step(param, grad.contiguous(), float(lr))
        return param
    return reference.sgd_step(param, grad, lr)


def fedavg_flat(models: torch.Tensor, weights: torch.Tensor) -> torch.Tensor:
    """``sum_k w_k * models[k]``; models ``[K,P]`` fp32, weights ``[K]`` (SURVEY K3)."""
    if _cuda(models):
        return _ext.require().fedavg_flat(models.contiguous(), weights.to(models.device, torch.float32).contiguous())
    return reference.fedavg_flat(models, weights)


def fedavg_apply(theta: torch.Tensor, models: torch.Tensor, weights: torch.Tensor, server_lr: float = 1.0) -> torch.Tensor:
    """``theta += server_lr * (sum_k w_k models[k] - theta)`` in place (reduce + scale + apply fused)."""
    if _cuda(theta):
        _ext.require().fedavg_apply(theta, models.contiguous(), weights.to(theta.device, torch.float32).contiguous(), float(server_lr))
        return theta
    return reference.fedavg_apply(theta, models, weights, server_lr)


def sigmoid_bce(z: torch.Tensor, y: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """(mean BCE(sigmoid(z), y), dL/dz) in one pass (SURVEY K9)."""
    if _cuda(z):
        loss, dz = _ext.require().sigmoid_bce(z.contiguous().float(), y.contiguous().float().view_as(z))
        return loss, dz
    return reference.sigmoid_bce(z, y)


def sse_loss(out: torch.Tensor, y: torch.Tensor, mean: bool = False) -> Tuple[torch.Tensor, torch.Tensor]:
    """(sum (out-y)^2 [/batch], gradient) (SURVEY K11)."""
    if _cuda(out):
        scale = 1.0 / out.shape[0] if mean else 1.0
        loss, dz = _ext.require().sse_loss(out.contiguous().float(), y.contiguous().float().view_as(out), scale)
        return loss, dz
    return reference.loss_and_dz(out, y, "mse" if mean else "sse", "none")


def softmax_xent(logits: torch.Tensor, labels: torch.Tensor, bf16_grad: bool = False) -> Tuple[torch.Tensor, torch.Tensor]:
    """(mean softmax cross-entropy, dL/dlogits) in one pass (SURVEY K10)."""
    if _cuda(logits):
        loss, dl = _ext.require().softmax_xent(logits.contiguous(), labels.contiguous().long().view(-1), bool(bf16_grad))
        return loss, dl
    loss, dl = reference.softmax_xent(logits, labels)
    return loss, (dl.to(torch.bfloat16) if bf16_grad else dl)


def eval_binary(p: torch.Tensor, y: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """(sum BCE, #correct round(p)==y) (SURVEY K15; reference ``evaluate`` cf.py:233-253)."""
    if _cuda(p):
        loss, correct = _ext.require().eval_binary(p.contiguous().float().view(-1), y.contiguous().float().view(-1))
        return loss, correct
    return reference.eval_binary(p, y)


def argmax_rows(x: torch.Tensor) -> torch.Tensor:
    """``x.argmax(1, keepdim=True)`` (SURVEY K16; reference inference fc.py:252-256)."""
    if _cuda(x):
        return _ext.require().argmax_rows(x.contiguous().float())
    return reference.argmax_rows(x)


def minmax_scale(x: torch.Tensor) -> torch.Tensor:
    """Column-wise scale to [0,1] (SURVEY K13; reference ``MinMaxScaler`` ds.py:31-32)."""
    if _cuda(x):
        return _ext.require().minmax_scale(x.contiguous().float())
    lo = x.min(0).values
    rng = x.max(0).values - lo
    rng = torch.where(rng == 0, torch.ones_like(rng), rng)
    return (x - lo) / rng


def device_permutation(n: int, rows: int, seed: int, device) -> torch.Tensor:
    """int32 ``[rows, n]`` keyed random permutations generated on the device (SURVEY K14).  A
    4-round Feistel bijection with cycle walking: every index is computed independently, so no
    H2D traffic and no serial Fisher-Yates.  CPU: ``reference.make_permutation``."""
    device = torch.device(device)
    if device.type == "cuda":
        return _ext.require().feistel_permutation(int(n), int(rows), int(seed), device)
    return reference.make_permutation(n, rows, seed)


def fp32_to_bf16(x: torch.Tensor) -> torch.Tensor:
    if _cuda(x):
        return _ext.require().fp32_to_bf16(x.contiguous())
    return x.to(torch.bfloat16)


def l2_flush(buf: torch.Tensor) -> None:
    """Overwrite a >L2-sized buffer (bench hygiene between timed iterations)."""
    if _cuda(buf):
        _ext.require().l2_flush(buf)
    else:
        buf.fill_(1.0)


from .linear import gemm_bf16, linear_forward, transpose_bf16, bias_sgd_from_partials  # noqa: E402,F401

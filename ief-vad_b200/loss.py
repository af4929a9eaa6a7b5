"""Drop-in for the reference's `train.loss.CLAS2` (train/loss.py:18-30) on the GPU: sigmoid, per-row top-k
(k = int(len/16 + 1)) mean and BCE in two kernels, k taken from the device `lengths` (no per-row host sync,
no O(B^2) torch.cat); and `train_loss`, the whole loss the reference's training loop builds from the module's outputs."""
from __future__ import annotations

from typing import NamedTuple

import torch

from . import ops


def CLAS2(logits: torch.Tensor, labels: torch.Tensor, lengths: torch.Tensor, device=None) -> torch.Tensor:
    """Same arguments as the reference; `device` is accepted and ignored (the tensors' device is used).  With a
    `logits` that requires grad the result carries a grad_fn (train.Clas2Fn: the top-k scatter of the BCE gradient),
    so `loss.backward()` of train/ucf_train.py:105 works."""
    if torch.is_grad_enabled() and logits.requires_grad:
        from .train import Clas2Fn
        return Clas2Fn.apply(logits, labels, lengths)
    loss, _ = ops.clas2(logits, labels, lengths)
    return loss


class TrainLoss(NamedTuple):
    """The parts of the training loss, each a 0-dim fp32 device tensor (log them without a host sync)."""
    total: torch.Tensor
    classification: torch.Tensor
    regulariser: torch.Tensor
    kl: torch.Tensor


def train_loss(outputs, labels: torch.Tensor, lengths: torch.Tensor, nu: float, reg_weight: float = 1.0,
               kl_weight: float = 1.0) -> TrainLoss:
    """The loss of train/ucf_train.py:73-102 from the module's output dict, in the kernels of csrc/train_loss.cu:

        total = CLAS2(logits, labels, lengths) + reg_weight * loss_reg + kl_weight * loss_kl
        loss_reg = mean(1 - cosine_similarity(normalize(image_mu), normalize(event_mu)))
                   + mean |norm(image_mu) - norm(event_mu)|
        loss_kl  = -0.5 mean(1 + eli - image_mu^2 - exp(eli)) - 0.5 mean(1 + ele - event_mu^2 - exp(ele)),
                   el = logvar + log(nu / (nu + 1))

    with the means over every row, pad rows included, as the loop computes them.  `nu` is the loop's
    `model.temporal.nu` (a number), whatever the noise model; the UCF loop's weights are 1 and 1.  With grad enabled
    and any of the five output tensors requiring grad the result is differentiable (train.TrainLossFn); otherwise only
    the forward kernels run.  All tensors must be on the GPU."""
    ts = tuple(outputs[k] for k in ("logits", "image_mu", "event_mu", "image_logvar", "event_logvar"))
    consts = (float(nu), float(reg_weight), float(kl_weight))
    if torch.is_grad_enabled() and any(t.requires_grad for t in ts):
        from .train import TrainLossFn
        return TrainLoss(*TrainLossFn.apply(*ts, labels, lengths, *consts))
    scalars, _ = ops.train_loss_fwd(ts[0], labels, lengths, *ts[1:], *consts)
    return TrainLoss(*scalars)

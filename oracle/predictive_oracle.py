"""CPU oracle for the VSMask PredictiveModel (SURVEY.md §8a row P).  TEST INFRASTRUCTURE ONLY.

Functional PyTorch restatement (fp32 or fp64) of ``/root/reference/models/predictive_model.py``:
  DownSamplingBlock  :6-28   ReflectionPad2d(1) -> Conv2d 3x3 (stride) -> BatchNorm2d -> PReLU(1 param)
  UpSamplingBlock    :30-51  ConvTranspose2d 3x3 stride 2 padding 0 -> LeakyReLU(0.2)
  PredictiveModel    :53-110 7 down blocks, 5 up blocks, tanh
Only ``tests/`` and bench legs may import it.  Pinned by executing the unmodified reference module
(loaded by file path: ``models.py`` shadows the ``models/`` directory, SURVEY §2 #8) in
tests/test_oracle_vs_reference.py, and on every run by tests/golden/vsmask_predictive.npz (tests/tools/make_golden.py).
"""
from __future__ import annotations

import math
from collections import OrderedDict
from typing import Dict, Optional, Tuple

import torch
import torch.nn.functional as F
from torch import Tensor

from attack_vc_b200.synthetic import PM_DOWN, PM_UP, pm_make_state_dict, pm_param_shapes  # noqa: F401,E402  (seeded generators only)

BN_EPS = 1e-5
BN_MOMENTUM = 0.1


def pm_forward(sd: Dict[str, Tensor], x: Tensor, training: bool = False,
               new_stats: Optional[Dict[str, Tensor]] = None) -> Tensor:
    """PredictiveModel.forward (predictive_model.py:87-110).  x [B,1,F,T] -> [B,1,F',T'].
    training=True uses batch statistics (the trainers call model.train(), train_predictive.py:64);
    the running-statistics update PyTorch performs as a side effect is returned in ``new_stats``."""
    h = x
    for i, (_, _, stride) in enumerate(PM_DOWN):
        p = f"down_blocks.{i}.conv."
        h = F.pad(h, (1, 1, 1, 1), mode="reflect")                               # ReflectionPad2d, :20-21
        h = F.conv2d(h, sd[p + "1.weight"], sd[p + "1.bias"], stride=stride)     # :22
        rm, rv = sd[p + "2.running_mean"].clone(), sd[p + "2.running_var"].clone()
        h = F.batch_norm(h, rm, rv, sd[p + "2.weight"], sd[p + "2.bias"], training=training,
                         momentum=BN_MOMENTUM, eps=BN_EPS)                        # :23
        if training and new_stats is not None:
            new_stats[p + "2.running_mean"], new_stats[p + "2.running_var"] = rm, rv
        h = F.prelu(h, sd[p + "3.weight"])                                       # :24
    for i in range(len(PM_UP)):
        p = f"up_blocks.{i}.conv_transpose.0."
        h = F.conv_transpose2d(h, sd[p + "weight"], sd[p + "bias"], stride=2)    # :46
        h = F.leaky_relu(h, 0.2)                                                 # :47
    return torch.tanh(h)                                                         # :108


def pm_out_shape(H: int, W: int) -> Tuple[int, int]:
    for _, _, (sh, sw) in PM_DOWN:
        H, W = (H + 2 - 3) // sh + 1, (W + 2 - 3) // sw + 1
    for _ in PM_UP:
        H, W = (H - 1) * 2 + 3, (W - 1) * 2 + 3
    return H, W


def pm_train_step(sd: Dict[str, Tensor], x: Tensor) -> Dict[str, object]:
    """One training forward/backward with the loss BASELINE config 5 names (SURVEY §8d):
    loss = out.square().mean(); returns loss, output, gradients of every parameter and of x."""
    params = {k: v.detach().clone().requires_grad_(True) for k, v in sd.items()
              if v.dtype.is_floating_point and "running" not in k}
    full = dict(sd)
    full.update(params)
    xin = x.detach().clone().requires_grad_(True)
    stats: Dict[str, Tensor] = {}
    out = pm_forward(full, xin, training=True, new_stats=stats)
    loss = out.square().mean()
    loss.backward()
    return {"loss": loss.detach(), "out": out.detach(), "grads": {k: v.grad.detach() for k, v in params.items()},
            "grad_x": xin.grad.detach(), "new_stats": stats}

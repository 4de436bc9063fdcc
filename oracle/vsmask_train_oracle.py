"""CPU oracle for the VSMask predictor training step (SURVEY.md §8f rank 3).  TEST INFRASTRUCTURE ONLY.

Restates the loop body of ``/root/reference/train_predictive.py:92-126`` with
``/root/reference/utils/audio.py:77-116`` (apply_weighted_constraint), ``torch.optim.Adam(model.parameters(), lr)``
(:57) and ``model.train()`` (:64), on top of the functional PredictiveModel of ``oracle/predictive_oracle.py``.

The reference loop cannot run as shipped (SURVEY §2 #8): ``perturbed_mels[:, :, :, fs:fe] += predicted[:, :, :, :fe-fs]``
adds a [B,1,95,63] prediction to a [B,1,80,63] slice (:102) and ``apply_weighted_constraint`` unpacks a 4-D tensor into
three names (utils/audio.py:93).  Two repairs are DEFINED here (and mirrored by ``avc_pm_trainer_step``):
  1. the prediction is cropped to its first F mel rows: ``predicted[:, :, :F, :fe-fs]``;
  2. the constraint is applied to ``perturbation.squeeze(1)`` (its mel axis is then dim 1, as the method expects).
``speaker_encoder`` is AdaIN-VC's SpeakerEncoder on ``mel.squeeze(1)`` (the script's DummySpeakerEncoder is a
placeholder, train_predictive.py:198-213), as for the universal header.

Pinned by tests/test_oracle_vs_reference.py: the same step driven through the reference's own PredictiveModel module
and the reference's own apply_weighted_constraint source (extracted from utils/audio.py: torchaudio is not installed, so
the module itself cannot be imported) is bit-identical; on every run by tests/golden/vsmask_train.npz.  Only ``tests/``
and bench legs may import this file.
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional, Sequence, Tuple

import torch
from torch import Tensor

from oracle.predictive_oracle import pm_forward


def weighted_constraint(perturbation: Tensor, epsilon1: float = 0.1, epsilon2: float = 0.05, epsilon3: float = 0.08) -> Tensor:
    """MelSpectrogramConverter.apply_weighted_constraint (utils/audio.py:77-116) on [B, F, T]."""
    _, freq_dim, _ = perturbation.shape                                     # :93
    low_end, high_start = int(freq_dim * 0.3), int(freq_dim * 0.7)          # :96-97
    return torch.cat([torch.clamp(perturbation[:, :low_end, :], -epsilon1, epsilon1),          # :105
                      torch.clamp(perturbation[:, low_end:high_start, :], -epsilon2, epsilon2),  # :106
                      torch.clamp(perturbation[:, high_start:, :], -epsilon3, epsilon3)], dim=1)  # :107-114


def perturb(source_mels: Tensor, predicted: Tensor, future_steps: int, eps: Sequence[float],
            constraint: Callable = weighted_constraint) -> Tensor:
    """train_predictive.py:95-111 with the two repairs of the module docstring.  source_mels [B,1,F,T]."""
    F, T = source_mels.shape[2], source_mels.shape[3]
    perturbed = source_mels.clone()                                                             # :100
    future_end = min(future_steps + predicted.shape[-1], T)                                     # :101
    perturbed[:, :, :, future_steps:future_end] += predicted[:, :, :F, :future_end - future_steps]   # :102 (+ crop)
    weighted = constraint((perturbed - source_mels).squeeze(1), eps[0], eps[1], eps[2]).unsqueeze(1)  # :105-110
    return source_mels + weighted                                                               # :111


def train_steps(sd: Dict[str, Tensor], speaker_encoder: Callable[[Tensor], Tensor], batches: Sequence[Tuple[Tensor, Tensor]],
                lr=1e-3, future_steps: int = 10, eps: Sequence[float] = (0.1, 0.05, 0.08), lambda_param: float = 0.5,
                inv_norm: Optional[float] = None, record_grads: bool = False) -> Dict[str, object]:
    """Runs ``len(batches)`` optimiser steps from the state dict ``sd`` (not modified).  ``lr`` is a float or one value
    per step (the reference's ReduceLROnPlateau changes it between epochs, :58-60,131).  Returns the losses, the final
    state dict (parameters + BatchNorm running statistics), the Adam moments and, optionally, every step's gradients."""
    state = {k: v.detach().clone() for k, v in sd.items()}
    names = [k for k, v in state.items() if v.dtype.is_floating_point and "running" not in k]
    params = {k: state[k].requires_grad_(True) for k in names}
    opt = torch.optim.Adam([params[k] for k in names], lr=lr if isinstance(lr, float) else lr[0])       # :57
    mse = torch.nn.functional.mse_loss if inv_norm is None else (lambda a, b: (a - b).square().sum() * inv_norm)
    enc = lambda m: speaker_encoder(m.squeeze(1))                                                       # noqa: E731
    losses: List[float] = []
    grads: List[Dict[str, Tensor]] = []
    for i, (source_mels, target_mels) in enumerate(batches):
        if not isinstance(lr, float):
            for g in opt.param_groups:
                g["lr"] = lr[i]
        stats: Dict[str, Tensor] = {}
        predicted = pm_forward(state, source_mels, training=True, new_stats=stats)                      # :64,92
        perturbed = perturb(source_mels, predicted, future_steps, eps)                                  # :95-111
        e_src, e_tgt, e_per = enc(source_mels), enc(target_mels), enc(perturbed)                        # :114-116
        loss = mse(e_per, e_tgt) - lambda_param * mse(e_per, e_src)                                     # :119-122
        opt.zero_grad()                                                                                 # :125
        loss.backward()                                                                                 # :126
        if record_grads:
            grads.append({k: params[k].grad.detach().clone() for k in names})
        opt.step()                                                                                      # :127
        for k, v in stats.items():
            state[k] = v.detach()
        losses.append(float(loss.detach()))
    out_sd = {k: v.detach().clone() for k, v in state.items()}
    moments = {k: (opt.state[params[k]]["exp_avg"].clone(), opt.state[params[k]]["exp_avg_sq"].clone()) for k in names
               if params[k] in opt.state}
    return {"losses": torch.tensor(losses, dtype=torch.float64), "state": out_sd, "moments": moments, "grads": grads}

"""Batch sharding of the attack loop over the GPUs of one box (SURVEY.md §8e).

Utterances are independent (no BatchNorm in AdaIN-VC, InstanceNorm and pooling are per utterance),
so a batch is split into contiguous slices, one per rank, weights replicated, and NO collective runs
inside the loop.  The only coupling is the MSE normaliser: ``nn.MSELoss()`` averages over the batch
too (attack_utils.py:32,70,114), and Adam is not scale invariant at these gradient magnitudes
(SURVEY §5), so every rank passes the GLOBAL 1/(B_total*D).  After the loop the perturbed utterances
are all-gathered and the per-iteration loss partial sums all-reduced (NCCL on GPUs; gloo in the CPU
tests of this host logic).
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist
from torch import Tensor


def shard_bounds(n: int, world: int, rank: int) -> Tuple[int, int]:
    """Contiguous slice [lo, hi) of n utterances owned by ``rank``; the first n % world ranks get one
    extra.  Empty slices are legal (world > n)."""
    base, extra = divmod(n, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def global_inv_norm(kind: str, B_total: int, c_emb: int, c_mel: int, T_out: int) -> float:
    """1 / (number of elements the reference's MSELoss averages over) for the WHOLE batch:
    emb / fb compare embeddings [B, c_emb]; e2e compares converted mels [B, c_mel, T_out]."""
    d = c_emb if kind in ("emb", "fb") else c_mel * T_out
    return 1.0 / (float(B_total) * d)


AttackFn = Callable[..., Tuple[Tensor, Dict[str, Optional[Tensor]]]]


def sharded_attack(attack: AttackFn, kind: str, vc_tgt: Tensor, adv_tgt: Tensor, eps: float, n_iters: int,
                   inv_norm: float, vc_src: Optional[Tensor] = None, w0: Optional[Tensor] = None,
                   group=None) -> Tuple[Tensor, Tensor]:
    """Run ``attack`` on this rank's slice of the (replicated) batch and return the full perturbed
    batch plus the per-iteration loss of the whole batch on every rank.

    ``attack(kind, vc_tgt, adv_tgt, eps, n_iters, vc_src=, w0=, inv_norm=, want_loss=True)`` is
    ``Engine.attack`` on a GPU; tests inject a CPU stand-in to exercise this plumbing under gloo."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    B = vc_tgt.shape[0]
    lo, hi = shard_bounds(B, world, rank)
    losses = torch.zeros(n_iters, dtype=torch.float32, device=vc_tgt.device)
    if hi > lo:
        sl = slice(lo, hi)
        adv, info = attack(kind, vc_tgt[sl], adv_tgt[sl], eps, n_iters,
                           vc_src=None if vc_src is None else vc_src[sl], w0=None if w0 is None else w0[sl],
                           inv_norm=inv_norm, want_loss=True)
        losses = info["losses"].to(torch.float32)
    else:
        adv = vc_tgt[0:0]
    return gather_shards(adv, losses, B, group=group)


def gather_shards(adv_local: Tensor, losses_local: Tensor, B_total: int, group=None) -> Tuple[Tensor, Tensor]:
    """The one collective step of a sharded attack, run AFTER the loop: all_gather of the perturbed utterances
    (equal-sized padded slots; slices differ by at most one utterance) and all_reduce(sum) of the per-iteration loss
    partial sums (each already scaled by the global normaliser).  NCCL over NVLink on GPUs, gloo in the CPU tests."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if world == 1:
        return adv_local, losses_local
    cap = -(-B_total // world)
    slot = torch.zeros((cap,) + tuple(adv_local.shape[1:]), dtype=adv_local.dtype, device=adv_local.device)
    slot[: adv_local.shape[0]] = adv_local
    full = torch.empty((world * cap,) + tuple(adv_local.shape[1:]), dtype=adv_local.dtype, device=adv_local.device)
    dist.all_gather(list(full.chunk(world)), slot, group=group)     # views of one buffer: no copy after the collective
    parts = []
    for r in range(world):
        a, b = shard_bounds(B_total, world, r)
        parts.append(full[r * cap: r * cap + (b - a)])
    losses = losses_local.to(torch.float32).clone()
    dist.all_reduce(losses, op=dist.ReduceOp.SUM, group=group)
    return (torch.cat(parts, dim=0) if B_total % world else full), losses


def sharded_attack_shards(attack: AttackFn, kind: str, vc_tgt_local: Tensor, adv_tgt_local: Tensor, eps: float, n_iters: int,
                          B_total: int, inv_norm: float, vc_src_local: Optional[Tensor] = None,
                          w0_local: Optional[Tensor] = None, group=None) -> Tuple[Tensor, Tensor]:
    """``sharded_attack`` for callers that already hold only THEIR slice (rows ``shard_bounds(B_total, world, rank)`` of
    the global batch): nothing is replicated -- BASELINE configs[3] is 3 x 671 MB of inputs in total, 84 MB per rank.
    Returns the full perturbed batch and the whole-batch loss curve on every rank."""
    adv, info = attack(kind, vc_tgt_local, adv_tgt_local, eps, n_iters, vc_src=vc_src_local, w0=w0_local,
                       inv_norm=inv_norm, want_loss=True)
    return gather_shards(adv, info["losses"], B_total, group=group)


def sharded_header_optimize(engine, source_mel: Tensor, target_mel: Tensor, num_iterations: int, epsilon: float = 0.1,
                            lambda_param: float = 0.5, lr: float = 1e-3, header0: Optional[Tensor] = None, group=None):
    """UniversalPerturbationHeader.optimize (models/header_model.py:25-68) with the batch sharded over the ranks.
    The header is shared by ALL utterances, so this is the one workload with a per-iteration collective: every
    rank runs forward/backward on its slice, the partial header gradients (80*T floats, 32 KB) are all-reduced,
    then every rank applies the same Adam step.  ``engine`` is an ``Engine`` (or a stand-in with ``header_begin``)."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    B = source_mel.shape[0]
    lo, hi = shard_bounds(B, world, rank)
    if hi <= lo:
        raise ValueError("sharded_header_optimize needs at least one utterance per rank")
    inv = 1.0 / (float(B) * 128)
    sess = engine.header_begin(source_mel[lo:hi], target_mel[lo:hi], num_iterations, epsilon, lambda_param, lr,
                               header0=header0, inv_norm=inv, want_loss=True)
    for _ in range(int(num_iterations)):
        sess.grad_half()
        if world > 1:
            dist.all_reduce(sess.grad, op=dist.ReduceOp.SUM, group=group)
        sess.apply_half()
    header, info = sess.end()
    losses = info["losses"].clone()
    if world > 1:
        dist.all_reduce(losses, op=dist.ReduceOp.SUM, group=group)
    return header, losses


def sharded_defend(defender, vc_tgt: Sequence[Tensor], adv_tgt: Tensor, group=None, **kw) -> List[Tensor]:
    """``defender.defend(vc_tgt, adv_tgt, **kw)`` with the utterances split into contiguous slices, one per rank
    (``shard_bounds``).  No collective runs during the work: given the per-utterance normaliser ``Defender`` uses, the
    utterances are independent.  At the end ONE gather of the variable-length waveforms (lengths, then a padded
    all-gather; NCCL on GPUs) returns every defended waveform, in input order, on every rank.  Each rank draws the
    initial noise of its slice from its own RNG."""
    if kw.get("return_mels"):
        raise ValueError("sharded_defend gathers waveforms only (return_mels is not supported)")
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    B = len(vc_tgt)
    lo, hi = shard_bounds(B, world, rank)
    local = list(defender.defend(list(vc_tgt[lo:hi]), adv_tgt, **kw)) if hi > lo else []
    return gather_varlen(local, B, defender.device, group=group)


def gather_varlen(local: Sequence[Tensor], B_total: int, device, group=None) -> List[Tensor]:
    """All-gather of 1-D tensors of different lengths, rank r holding items ``shard_bounds(B_total, world, r)``: one
    all-gather of the lengths, one of equal-sized padded slots."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if world == 1:
        return list(local)
    cap = max(-(-B_total // world), 1)
    lens = torch.zeros(cap, dtype=torch.int64, device=device)
    if local:
        lens[: len(local)] = torch.tensor([int(w.numel()) for w in local], dtype=torch.int64)
    all_lens = torch.empty(world * cap, dtype=torch.int64, device=device)
    dist.all_gather(list(all_lens.chunk(world)), lens, group=group)
    L = max(int(all_lens.max()), 1)
    slot = torch.zeros(cap, L, dtype=torch.float32, device=device)
    for k, w in enumerate(local):
        slot[k, : w.numel()] = w
    full = torch.empty(world * cap, L, dtype=torch.float32, device=device)
    dist.all_gather(list(full.chunk(world)), slot, group=group)
    n = all_lens.tolist()
    out = []
    for r in range(world):
        a, b = shard_bounds(B_total, world, r)
        out.extend(full[r * cap + k, : n[r * cap + k]] for k in range(b - a))
    return out

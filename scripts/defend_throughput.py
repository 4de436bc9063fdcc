"""Defended utterances per second, device-resident waveform to device-resident waveform (attack_vc_b200.Defender).

  python scripts/defend_throughput.py --attack emb --utterances 512 --frames 512 --gpus 8

Every GPU defends ``--utterances`` seeded synthetic waveforms of ``hop (F - 1)`` samples (tones plus noise, like
tests/test_audio_gpu.py::tone; ``--ragged`` spreads the frame counts over +-25 % of F) with the synthetic model (seed 0)
and speaker statistics taken from the synthetic corpus's own mels: one ragged front-end call, the attacks grouped by
length, one ragged back-end call.  With ``--gpus N`` one process per GPU defends its own slice and the waveforms are
all-gathered at the end (NCCL), inside the timed region.  One warm-up defence at the timed shapes, then one timed
defence: host clock around a call that ends in torch.cuda.synchronize(), CUDA events per stage.  Prints one JSON line.
``--mixed-lengths`` runs the attacks as ragged calls over chunks of the length-sorted utterances (``defend(...,
mixed_lengths=True)``) instead of grouping them by length.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import socket
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from attack_vc_b200 import Defender  # noqa: E402
from attack_vc_b200.audio import AudioEngine  # noqa: E402
from attack_vc_b200.synthetic import SYNTH_CONFIG, ParamTree  # noqa: E402

SR, HOP = 24000, 300


def tone(n: int, seed: int, device) -> torch.Tensor:
    """tests/test_audio_gpu.py::tone, generated on the device (a seeded synthetic input, not part of what is timed)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    noise = torch.randn(n, generator=g, dtype=torch.float64).to(device)
    t = torch.arange(n, device=device, dtype=torch.float64) / SR
    w = (0.3 * torch.sin(2 * math.pi * 220 * t) + 0.15 * torch.sin(2 * math.pi * 1333 * t + 0.3)
         + 0.05 * torch.sin(2 * math.pi * 5100 * t) + 0.02 * noise)
    return (w * torch.hann_window(n, periodic=False, dtype=torch.float64, device=device) ** 0.25).float()


def frame_counts(B: int, F: int, ragged: bool, seed: int):
    if not ragged:
        return [F] * B
    g = torch.Generator().manual_seed(seed)
    return [max(16, int(round(F * (1 + 0.25 * (2 * float(u) - 1))))) for u in torch.rand(B, generator=g)]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return torch.cuda.get_device_name(0), (q.stdout.strip().splitlines() or [q.stderr.strip()])[0]


def run(rank: int, world: int, port: int, args, q):
    import torch.distributed as dist
    from attack_vc_b200.distributed import gather_varlen, shard_bounds
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    if world > 1:
        dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    B_total = args.utterances * world
    lo, hi = shard_bounds(B_total, world, rank)
    frames = frame_counts(B_total, args.frames, args.ragged, 1)
    wavs = [tone(HOP * (frames[i] - 1), 1000 + i, dev) for i in range(lo, hi)]
    adv = tone(HOP * (args.frames - 1), 7, dev)
    src = tone(HOP * (args.frames - 1), 8, dev) if args.attack != "emb" else None
    audio = AudioEngine(device=dev)
    corpus = audio.wav2mel_varlen([tone(HOP * (args.frames - 1), 2000 + i, dev) for i in range(16)])
    allm = torch.cat(corpus)
    mean, std = allm.mean(0), allm.std(0).clamp_min(1e-3)
    d = Defender(ParamTree(SYNTH_CONFIG, seed=0).to(dev), mean, std, audio=audio)

    def once():
        torch.manual_seed(rank)
        out = d.defend(wavs, adv, attack_type=args.attack, n_iters=args.iters, vc_src=src, griffin_lim_iters=args.gl_iters,
                       mixed_lengths=args.mixed_lengths)
        if world > 1:
            out = gather_varlen(out, B_total, dev)
        torch.cuda.synchronize(dev)
        return out

    once()                                                             # warm-up at the timed shapes
    if world > 1:
        dist.barrier()
    l0 = d.kernel_launches
    t0 = time.perf_counter()
    out = once()
    sec = time.perf_counter() - t0
    launches = d.kernel_launches - l0
    assert len(out) == B_total and all(bool(torch.isfinite(w).all()) for w in out[:4])
    res = dict(rank=rank, seconds=sec, stages_ms=d.last_stage_ms, kernel_launches=launches, utterances=hi - lo)
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, res)
        dist.destroy_process_group()
    else:
        gathered = [res]
    if rank == 0:
        q.put(gathered)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--attack", choices=["emb", "e2e", "fb"], default="emb")
    ap.add_argument("--utterances", type=int, default=512, help="utterances per GPU")
    ap.add_argument("--frames", type=int, default=512)
    ap.add_argument("--ragged", action="store_true")
    ap.add_argument("--mixed-lengths", action="store_true", help="ragged attack calls over length-sorted chunks")
    ap.add_argument("--iters", type=int, default=1500)
    ap.add_argument("--gl-iters", type=int, default=100)
    ap.add_argument("--gpus", type=int, default=1)
    args = ap.parse_args()
    if not torch.cuda.is_available() or torch.cuda.device_count() < args.gpus:
        raise SystemExit(f"needs {args.gpus} CUDA device(s); found {torch.cuda.device_count() if torch.cuda.is_available() else 0}")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    procs = [ctx.Process(target=run, args=(r, args.gpus, port, args, q)) for r in range(args.gpus)]
    for p in procs:
        p.start()
    import queue
    while True:                                                        # a rank that dies must not leave this waiting
        try:
            ranks = q.get(timeout=5)
            break
        except queue.Empty:
            if any(p.exitcode not in (None, 0) for p in procs):
                for p in procs:
                    p.kill()
                raise SystemExit("a rank failed (see its traceback above)")
    for p in procs:
        p.join()
        if p.exitcode != 0:
            raise SystemExit(f"a rank exited with {p.exitcode}")
    name, limits = gpu_info()
    sec = max(r["seconds"] for r in ranks)
    total = sum(r["utterances"] for r in ranks)
    print(json.dumps(dict(
        metric="defended utterances/s", attack=args.attack, utterances_per_gpu=args.utterances, frames=args.frames,
        ragged=args.ragged, mixed_lengths=args.mixed_lengths, iters=args.iters, gl_iters=args.gl_iters, gpus=args.gpus, seconds=round(sec, 4),
        utt_per_s_total=round(total / sec, 3), utt_per_s_per_gpu=round(total / sec / args.gpus, 3),
        stages_ms_rank0={k: round(v, 3) for k, v in ranks[0]["stages_ms"].items()},
        kernel_launches_rank0=ranks[0]["kernel_launches"], gpu=name, power_limit_and_max_sm_clock=limits)))


if __name__ == "__main__":
    main()

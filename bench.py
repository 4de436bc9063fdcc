#!/usr/bin/env python
"""bench.py -- attack iterations/s of the attack-vc perturbation loop on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload e2e|fb|emb|pm|vsmask|gl]
                    [--dump-outputs DIR]

A *step* is one attack iteration (adv = x + eps*tanh(w); forward; loss; backward; Adam) over one
batch of synthetic 80-bin mel utterances.  Default workload = BASELINE.json configs[1]: e2e_attack,
1 utterance of 80 x 256 frames per GPU, random-init AdaIN-VC weights.  Multi-GPU: one process per
GPU (torchrun), independent utterances per rank, no collective in the loop ("weak" scaling); the
perturbed outputs and loss curves are gathered with NCCL after the loop.

Numbers in the JSON line
  value     iterations/s x utterances, inputs resident in HBM, CUDA events around exactly K steps
            (graph replays of the captured iteration), max over ranks.
  e2e       same metric through the drop-in public API attack_utils.<kind>_attack(...) with pinned
            HOST tensors: H2D copies, target/invariant computation, K iterations, D2H of the result
            all inside the timed region.
  roofline  conv kernels (the dominant kernel class): algorithmic FLOPs / per-launch CUDA-event time
            from one eagerly launched iteration, against MEASURED_PEAKS.json.
  cpu_baseline  the oracle (PyTorch CPU restatement of the reference loop, incl. its wgrad and
            per-iteration content-encoder work) on this box's host cores, bounded sample.
`--impl reference` times that CPU loop alone (the reference is Python/PyTorch and is not part of this
repository; the oracle is bit-identical to it -- tests/test_oracle_vs_reference.py).

`--dump-outputs DIR` writes, after the timed steps, what the timed path returned for its last step as
DIR/<name>.npy (float32; rank 0).  Inputs and weights are seeded, so two builds run with the same
arguments can be compared output for output.  Arrays are sampled along their first axis with a fixed
seed where the files would otherwise exceed 64 MB in all.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
os.environ.setdefault("TQDM_DISABLE", "1")     # the drop-in keeps the reference's progress bar; keep stderr quiet here

import torch  # noqa: E402

WORKLOADS = {
    # name: (kind, utterances per GPU, frames, description)
    "e2e": ("e2e", 1, 256, "BASELINE configs[1]: e2e_attack, ContentEncoder+SpeakerEncoder+Decoder, 80x256, batch 1 per GPU"),
    "fb": ("fb", 64, 256, "BASELINE configs[2]: fb_attack, 80x256, batch 64 per GPU"),
    "emb": ("emb", 512, 512, "BASELINE configs[3]: emb_attack, 80x512, 512 utterances per GPU (4096 over 8)"),
    "pm": ("pm", 256, 100, "BASELINE configs[4]: VSMask predictive_model forward/backward, 80x100 windows, batch 256 per GPU"),
    "vsmask": ("vsmask", 256, 100, "SURVEY 8f rank 3: VSMask predictor training step (train_predictive.py:92-127), 80x100 windows, batch 256 per GPU"),
    "gl": ("gl", 16, 256, "SURVEY 8f rank 4: mel2wav with 100 Griffin-Lim iterations (data_utils.py:120-197), 80-mel x 256-frame utterances, batch 16 per GPU"),
}
KIND_NAMES = {0: "conv", 1: "norm", 2: "dense_tail", 3: "affine", 4: "loss", 5: "update", 6: "layout", 7: "copy"}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained"),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


DUMP_BYTES = 64 * 10**6


def dump_outputs(path: str, arrays: dict) -> None:
    """--dump-outputs: every tensor of `arrays` as path/<name>.npy in float32, all files together within DUMP_BYTES.
    An array over its share keeps a fixed, seeded subset of its rows (first axis; elements when one row is too big)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    items = sorted(arrays.items(), key=lambda kv: kv[1].numel())        # small arrays first: the big ones share the rest
    left = DUMP_BYTES
    for i, (name, t) in enumerate(items):
        a = t.detach().float().cpu().numpy().reshape(t.shape or (1,))
        share = left // (len(items) - i) - 4096                        # 4096: room for the .npy header
        if a.nbytes > share:
            if a[0].nbytes > share:
                a = a.reshape(-1)
            keep = np.sort(np.random.default_rng(0).choice(a.shape[0], share // a[0].nbytes, replace=False))
            a = a[keep]
        np.save(os.path.join(path, name + ".npy"), a)
        left -= os.path.getsize(os.path.join(path, name + ".npy"))
        print(f"bench.py: {path}/{name}.npy {list(a.shape)} of {list(t.shape)}", file=sys.stderr)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the timed region runs."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.12)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
            self.thread.join(timeout=1)

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def cpu_loop_rate(kind: str, B: int, T: int, budget_s: float, max_iters: int):
    """iterations/s of the oracle loop (== reference loop) on the host cores; bounded sample."""
    from oracle import adainvc_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    model = O.OracleAdaInVC(O.SYNTH_CONFIG, seed=0)
    inp = O.make_inputs(kind, B, T, seed=1)
    run = lambda n: O.run_attack(kind, model, inp["vc_tgt"], inp["adv_tgt"], 0.1, n, inp["w0"], vc_src=inp.get("vc_src"))
    run(2)                                  # warm-up (thread pool, mkldnn primitives)
    t0 = time.perf_counter(); run(3); t3 = time.perf_counter() - t0
    n = int(max(5, min(max_iters, budget_s / (t3 / 3))))
    t0 = time.perf_counter(); run(n); dt = time.perf_counter() - t0
    # run(n) also recomputes the two targets once; that is part of the reference's attack call
    return n * B / dt, cores, n, dt


def gpu_eager_baseline(kind: str, B: int, T: int, dev, budget_s: float = 8.0):
    """The "library bar" (SURVEY 8d, BASELINE.md 3.5): the SAME loop as the reference (oracle loop == reference loop)
    run by PyTorch eager on this B200 -- cuDNN / cuBLAS fp32 kernels, TF32 off -- with resident inputs.  Also tried once
    inside a CUDA graph (capturable Adam), which removes eager's launch overhead.  Checker / baseline code only."""
    from oracle import adainvc_oracle as O
    tf32 = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    out = {"what": "oracle loop (== reference loop) on cuda, PyTorch eager fp32, allow_tf32 = False", "torch": torch.__version__}
    try:
        model = O.OracleAdaInVC(O.SYNTH_CONFIG, seed=0).to(dev)
        inp = {k: v.to(dev) for k, v in O.make_inputs(kind, B, T, seed=1).items()}
        run = lambda n: O.run_attack(kind, model, inp["vc_tgt"], inp["adv_tgt"], 0.1, n, inp["w0"], vc_src=inp.get("vc_src"))
        run(3); torch.cuda.synchronize(dev)
        t0 = time.perf_counter(); run(5); torch.cuda.synchronize(dev); t5 = (time.perf_counter() - t0) / 5
        n = int(max(10, min(300, budget_s / max(t5, 1e-4))))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev); e0.record(); r = run(n); e1.record(); torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / n
        out.update({"value": B * 1e3 / ms, "unit": "utterance-iterations/s", "ms_per_step": ms, "iterations": n,
                    "loss_last": float(r["losses"][-1])})
        try:   # kernels per iteration: difference of two profiled runs of different length
            from torch.profiler import ProfilerActivity, profile

            def kernels(k):
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    run(k); torch.cuda.synchronize(dev)
                return sum(1 for ev in prof.events() if str(ev.device_type).endswith("CUDA"))
            out["launches_per_iter"] = (kernels(4) - kernels(2)) / 2.0
        except Exception as e:
            out["launches_per_iter"] = None; out["launches_error"] = str(e)[:120]
        try:   # the same iteration captured into a CUDA graph (whole-network capture, capturable Adam)
            x, at, src = inp["vc_tgt"], inp["adv_tgt"], inp.get("vc_src")
            mse = torch.nn.MSELoss()
            fwd = {"emb": lambda a: model.speaker_encoder(a), "e2e": lambda a: model.inference(src, a),
                   "fb": lambda a: model.speaker_encoder(model.inference(src, a))}[kind]
            with torch.no_grad():
                org = fwd(x); tgt = model.speaker_encoder(at) if kind in ("emb", "fb") else model.inference(src, at)
            w = inp["w0"].clone().requires_grad_(True)
            opt = torch.optim.Adam([w], capturable=True)

            side = torch.cuda.Stream(); side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(3):
                    opt.zero_grad(set_to_none=True)
                    o = fwd(x + 0.1 * w.tanh()); loss = mse(o, tgt) - 0.1 * mse(o, org); loss.backward(); opt.step()
            torch.cuda.current_stream().wait_stream(side)
            g = torch.cuda.CUDAGraph()
            opt.zero_grad(set_to_none=True)
            for prm in model.parameters():
                prm.grad = None
            with torch.cuda.graph(g):
                o = fwd(x + 0.1 * w.tanh()); loss = mse(o, tgt) - 0.1 * mse(o, org); loss.backward(); opt.step()
            for _ in range(3):
                g.replay()
            ng = int(max(20, min(2000, budget_s / 2 / max(ms / 1e3 / 4, 1e-5))))
            torch.cuda.synchronize(dev); e0.record()
            for _ in range(ng):
                g.replay()
            e1.record(); torch.cuda.synchronize(dev)
            msg = e0.elapsed_time(e1) / ng
            out["cuda_graph"] = {"value": B * 1e3 / msg, "ms_per_step": msg, "iterations": ng, "loss": float(loss)}
        except Exception as e:
            out["cuda_graph"] = {"error": str(e)[:200]}
    except Exception as e:
        out["error"] = str(e)[:200]
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = tf32
    return out


PM_GFLOP_FWD, PM_GFLOP_FWD_BWD = 0.2045, 0.6111        # per 80x100 window, SURVEY 8d
# speaker-encoder work of one trainer step per window: three forwards + one dgrad pass = 4 x 2 x SE(T = 100) FLOP, SE(T) in MACs (SURVEY 8)
VSMASK_SE_GFLOP = 4 * 2 * (1011712 * 100 + 212992) / 1e9


def pm_cpu_rate(B: int, budget_s: float, vsmask: bool = False):
    """windows/s of the oracle training step (== reference module + autograd) on the host cores.  vsmask: the whole
    trainer step of train_predictive.py:92-127 (predictive model + 3 speaker-encoder passes + Adam)."""
    from oracle import predictive_oracle as P
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sd = P.pm_make_state_dict(0)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(B, 1, 80, 100, generator=g)
    if vsmask:
        from oracle import adainvc_oracle as O
        from oracle import vsmask_train_oracle as V
        se = O.OracleAdaInVC(O.SYNTH_CONFIG, seed=0)
        y = torch.randn(B, 1, 80, 100, generator=g)
        step = lambda: V.train_steps(sd, se.speaker_encoder, [(x, y)])      # noqa: E731
    else:
        step = lambda: P.pm_train_step(sd, x)                               # noqa: E731
    step()
    t0 = time.perf_counter(); step(); t1 = time.perf_counter() - t0
    n = int(max(2, min(50, budget_s / t1)))
    t0 = time.perf_counter()
    for _ in range(n):
        step()
    dt = time.perf_counter() - t0
    return n * B / dt, cores, n, dt


def pm_arm(args, rank, world, local):
    """BASELINE configs[4].  pm: one step = model.train(); out = model(x); out.square().mean().backward() on a batch of
    80x100 windows.  vsmask: one step = the reference's whole trainer iteration (train_predictive.py:92-127).
    Multi-GPU = data parallel as the config names it: every rank holds B windows of ONE global batch -- BatchNorm
    statistics over the global batch (all-reduce of the per-channel sums, 7 layers forward + 7 backward), global loss
    normaliser, one all-reduce of the 6.09 M parameter gradients per step -- NCCL through torch.distributed."""
    import torch.distributed as dist
    vsmask = args.workload == "vsmask"
    _, B, T, desc = WORKLOADS[args.workload]
    metric = "predictive_model windows/s (" + ("VSMask trainer step: forward, speaker loss, backward, Adam)" if vsmask else "train forward+backward)")
    if args.impl == "reference":
        if rank != 0:
            return
        rate, cores, n, dt = pm_cpu_rate(32, 20.0, vsmask)
        line = {"impl": "reference", "metric": metric, "value": rate, "unit": "windows/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * 32 / rate, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": desc, "windows_per_gpu": B, "window": "1x80x100"},
                "cpu_baseline": {"value": rate, "unit": "windows/s", "cores": cores, "kind": "port",
                                 "sample": f"{n} training steps of 32 windows, oracle (bit-identical to the reference pieces), {dt:.1f} s"},
                "e2e": {"value": rate, "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line), flush=True)
        return
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        sys.stdout.flush(); saved = os.dup(1); os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.all_reduce(torch.zeros(1, device=dev)); torch.cuda.synchronize(dev)
        finally:
            sys.stdout.flush(); os.dup2(saved, 1); os.close(saved)
    from attack_vc_b200.synthetic import pm_make_state_dict
    from attack_vc_b200.predictive import PredictiveEngine, PredictiveTrainer
    eng = PredictiveEngine({k: v.to(dev) for k, v in pm_make_state_dict(0).items()})
    eng.set_process_group(None, world)
    K, W = args.steps, max(args.warmup, 3)
    g = torch.Generator().manual_seed(3 + rank)
    host = torch.randn(B, 1, 80, T, generator=g).pin_memory()
    host_t = torch.randn(B, 1, 80, T, generator=g).pin_memory()
    x, y = host.to(dev), host_t.to(dev)
    se = trainer = None
    if vsmask:
        from attack_vc_b200 import Engine
        from attack_vc_b200.synthetic import SYNTH_CONFIG, ParamTree
        se = Engine(ParamTree(SYNTH_CONFIG, seed=0).to(dev))
        trainer = PredictiveTrainer(eng, se, batch_size=B, inv_norm=1.0 / (B * world * 128))

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def mx(v):
        if world == 1:
            return v
        t = torch.tensor([v], device=dev, dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX); return float(t.item())

    last = {}                                 # what the last train_step returned (--dump-outputs)

    def step(xs, ys):
        if vsmask:
            return trainer.step(xs, ys, lr=1e-3)
        r = eng.train_step(xs, reuse_buffers=True)
        if world > 1:
            dist.all_reduce(r["flat"])        # the gradients of the global batch: one 24.4 MB collective
        last.update(r)
        return r["loss"]
    launches_of = lambda: eng.kernel_launches + (se.kernel_launches if se is not None else 0)      # noqa: E731
    for _ in range(W):
        step(x, y)
    l0 = launches_of()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    with ClockSampler(local) as clk:
        e0.record()
        for _ in range(K):
            loss = step(x, y)
        e1.record()
        sync_all()
    ms = mx(e0.elapsed_time(e1))
    launches = launches_of() - l0
    value = K * B * world / (ms / 1e3)
    if args.dump_outputs and rank == 0:
        if vsmask:      # the step returns the loss; the weights and BatchNorm statistics it updated are read back
            state = trainer.state_dict()
            dump_outputs(args.dump_outputs, {"loss": loss, "state": torch.cat([v.reshape(-1) for v in state.values()])})
        else:
            dump_outputs(args.dump_outputs, {"loss": last["loss"], "out": last["out"], "grads": last["flat"],
                                             "new_stats": torch.cat([v.reshape(-1) for v in last["new_stats"].values()])})
    # eval forward alone
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fwd_rate = None
    if not vsmask:
        eng.forward(x); torch.cuda.synchronize(dev); a.record()
        for _ in range(max(3, K)):
            eng.forward(x)
        b.record(); torch.cuda.synchronize(dev)
        fwd_rate = max(3, K) * B * 1e3 / a.elapsed_time(b)
    # e2e: pinned host windows -> device, training step, loss back to the host, every step
    sync_all(); t0 = time.perf_counter()
    for _ in range(K):
        loss = step(host.to(dev, non_blocking=True), host_t.to(dev, non_blocking=True) if vsmask else None); lv = float(loss.cpu())
    e2e_ms = mx(1e3 * (time.perf_counter() - t0))
    peaks = load_peaks()
    gflop = PM_GFLOP_FWD_BWD + (VSMASK_SE_GFLOP if vsmask else 0.0)
    tf = value / world * gflop / 1e3
    dp = ("data parallel: BatchNorm over the global batch (all-reduce of per-channel sums, 7 layers forward + 7 backward), "
          "one all-reduce of the 6 088 904 parameter gradients per step, NCCL via torch.distributed") if world > 1 else "single device"
    line = {"metric": metric, "value": value, "unit": "windows/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": desc, "windows_per_gpu": B, "window": "1x80x100",
                       "loss": "mse(SE(perturbed), SE(target)) - 0.5 mse(SE(perturbed), SE(source)), Adam lr 1e-3" if vsmask else "out.square().mean()",
                       "multi_gpu": dp, "l2": "activations of one step (2.6 GB at batch 256) exceed L2"},
            "detail": {"eval_forward_windows_per_s_per_gpu": fwd_rate},
            "clocks": clk.summary(),
            "e2e": {"value": K * B * world / (e2e_ms / 1e3), "unit": "windows/s", "h2d_bytes_per_step": host.numel() * 4 * (2 if vsmask else 1), "d2h_bytes_per_step": 4,
                    "api": ("PredictiveTrainer.step" if vsmask else "PredictiveEngine.train_step") + "(pinned host windows) + loss.cpu() per step"},
            "gpu_launches": launches, "launches_per_step": launches / K,
            "roofline": {"bound": "tensor", "achieved": tf, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": tf / peaks["bf16_tflops"],
                         "traffic": None, "kernel": "whole step: conv2d_tc_kernel / wgrad_tc_kernel (TMA tensor loads + tcgen05, 3xTF32: the tensor pipe executes 3x the algorithmic FLOPs at the TF32 rate, "
                                   "i.e. 6 bf16-equivalents per FLOP) + BatchNorm / PReLU / reduction kernels" + (" + speaker-encoder tcgen05 convs" if vsmask else ""),
                         "algorithmic_gflop_per_window": gflop, "peak_source": peaks["source"] + ", bf16 dense burst"},
            "loss": lv}
    if world == 1 and not args.no_cpu_baseline:
        rate, cores, n, dt = pm_cpu_rate(32, 15.0, vsmask)
        line["cpu_baseline"] = {"value": rate, "unit": "windows/s", "cores": cores, "kind": "port",
                                "sample": f"{n} training steps of 32 windows, oracle (bit-identical to the reference pieces), {dt:.1f} s"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if trainer is not None:
        trainer.close(); se.close()
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def gl_cpu_rate(budget_s: float):
    """utterances/s of the numpy oracle's mel2wav (100 Griffin-Lim iterations, 256 frames) on the host cores."""
    from oracle import audio_oracle as A
    import numpy as np
    mel = np.random.default_rng(0).random((256, 80)).astype(np.float32)
    t0 = time.perf_counter(); A.mel2wav(mel, n_iter=100); t1 = time.perf_counter() - t0
    n = int(max(1, min(8, budget_s / t1)))
    t0 = time.perf_counter()
    for _ in range(n):
        A.mel2wav(mel, n_iter=100)
    dt = time.perf_counter() - t0
    return n / dt, os.cpu_count() or 1, n, dt


def gl_arm(args, rank, world, local):
    """SURVEY 8f rank 4: one step = mel2wav (inverse mel, 100 Griffin-Lim iterations, de-emphasis) of a batch of utterances.
    Multi-GPU: independent utterances per rank (replicas, no collective)."""
    import torch.distributed as dist
    _, B, F, desc = WORKLOADS["gl"]
    metric = "mel2wav reconstructions/s (100 Griffin-Lim iterations)"
    if args.impl == "reference":
        if rank != 0:
            return
        rate, cores, n, dt = gl_cpu_rate(20.0)
        print(json.dumps({"impl": "reference", "metric": metric, "value": rate, "unit": "utterances/s", "n_gpus": args.gpus, "steps": args.steps,
                          "warmup": args.warmup, "ms_per_step": 1e3 / rate, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                          "data": "synthetic", "config": {"workload": desc, "utterances_per_gpu": B, "frames": F},
                          "cpu_baseline": {"value": rate, "unit": "utterances/s", "cores": cores, "kind": "port",
                                           "sample": f"{n} utterances of 256 frames, numpy oracle (numpy.fft; librosa is not installed), {dt:.1f} s"},
                          "e2e": {"value": rate, "unit": "utterances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}), flush=True)
        return
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        sys.stdout.flush(); saved = os.dup(1); os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.all_reduce(torch.zeros(1, device=dev)); torch.cuda.synchronize(dev)
        finally:
            sys.stdout.flush(); os.dup2(saved, 1); os.close(saved)
    from attack_vc_b200.audio import AudioEngine
    eng = AudioEngine(device=dev)
    K, W = args.steps, max(args.warmup, 3)
    host = torch.rand(B, F, 80, generator=torch.Generator().manual_seed(5 + rank)).pin_memory()
    mel = host.to(dev)

    def mx(v):
        if world == 1:
            return v
        t = torch.tensor([v], device=dev, dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX); return float(t.item())
    for _ in range(W):
        eng.mel2wav(mel, n_iter=100)
    l0 = eng.kernel_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    with ClockSampler(local) as clk:
        e0.record()
        for _ in range(K):
            wav = eng.mel2wav(mel, n_iter=100)
        e1.record()
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
    ms = mx(e0.elapsed_time(e1))
    launches = eng.kernel_launches - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"wav": wav})
    t0 = time.perf_counter()
    for _ in range(K):
        w = eng.mel2wav(host.to(dev, non_blocking=True), n_iter=100).cpu()
    e2e_ms = mx(1e3 * (time.perf_counter() - t0))
    peaks = load_peaks()
    # algorithmic FLOPs: 201 transforms per utterance, each a [F, 2048] x [2048, 2050] real GEMM
    gflop = 201 * 2.0 * F * 2048 * 2050 / 1e9
    tf = K * B * gflop / (ms / 1e3) / 1e3
    line = {"metric": metric, "value": K * B * world / (ms / 1e3), "unit": "utterances/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": desc, "utterances_per_gpu": B, "frames": F, "n_fft": 2048, "hop_length": 300, "win_length": 1200,
                       "l2": "the operand planes of one iteration (4 x 16 x 256 x 2048 x 4 B = 134 MB) exceed L2"},
            "clocks": clk.summary(),
            "e2e": {"value": K * B * world / (e2e_ms / 1e3), "unit": "utterances/s", "h2d_bytes_per_step": host.numel() * 4, "d2h_bytes_per_step": int(w.numel()) * 4,
                    "api": "AudioEngine.mel2wav(pinned host mels) + waveform.cpu() per step"},
            "gpu_launches": launches, "launches_per_step": launches / K,
            "roofline": {"bound": "tensor", "achieved": tf, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": tf / peaks["bf16_tflops"], "traffic": None,
                         "kernel": "conv2d_tc_kernel as the DFT / inverse-DFT GEMM (TMA + tcgen05, 3xTF32: 6 bf16-equivalents per algorithmic FLOP; a dense DFT does ~70x the FLOPs of an FFT)",
                         "algorithmic_gflop_per_utterance": gflop, "peak_source": peaks["source"] + ", bf16 dense burst"}}
    if world == 1 and not args.no_cpu_baseline:
        rate, cores, n, dt = gl_cpu_rate(12.0)
        line["cpu_baseline"] = {"value": rate, "unit": "utterances/s", "cores": cores, "kind": "port",
                                "sample": f"{n} utterances of 256 frames, numpy oracle (numpy.fft; librosa is not installed), {dt:.1f} s"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def reference_arm(args, rank):
    kind, B, T, desc = WORKLOADS[args.workload]
    if rank != 0:
        return
    Bc = min(B, 8)        # batched workloads: CPU sub-batch of 8 utterances (SURVEY 8d)
    rate, cores, n, dt = cpu_loop_rate(kind, Bc, T, budget_s=20.0, max_iters=max(5, args.steps))
    sample = f"{n} iterations of {kind}_attack, {Bc} utterance(s) of 80x{T}, oracle loop (bit-identical to the reference loop), {dt:.1f} s"
    line = {
        "impl": "reference", "metric": "attack iterations/s (x utterances)", "value": rate, "unit": "utterance-iterations/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * Bc / rate, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": desc, "attack": kind, "utterances_per_gpu": B, "frames": T, "eps": 0.1},
        "cpu_baseline": {"value": rate, "unit": "utterance-iterations/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": "utterance-iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "ONE CPU process on rank 0 with all host cores, whatever --gpus says (the reference has no multi-process path): "
                "at N > 1 this is not N reference processes -- compare the N-GPU value with N x this only with that in mind",
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1500)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="e2e", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the batched side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1: every rate is the timed steps over their time")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the b200 path computed; it does not apply to --impl reference")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.workload == "gl":
        if args.impl != "reference" and not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; attack_vc_b200 has no CPU fallback (use --impl reference for the CPU loop)")
        gl_arm(args, rank, world, local)
        return
    if args.workload in ("pm", "vsmask"):
        if args.impl != "reference" and not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; attack_vc_b200 has no CPU fallback (use --impl reference for the CPU loop)")
        pm_arm(args, rank, world, local)
        return
    if args.impl == "reference":
        reference_arm(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; attack_vc_b200 has no CPU fallback (use --impl reference for the CPU loop)")

    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner on stdout when the communicator is created; the contract is ONE
        # JSON line there, so stdout is pointed at stderr until the communicator exists.
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize(dev)
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    from attack_vc_b200 import Engine
    from attack_vc_b200.synthetic import SYNTH_CONFIG, ParamTree, make_inputs
    import attack_utils as AU

    kind, B, T, desc = WORKLOADS[args.workload]
    K, W = args.steps, max(args.warmup, 3)
    model = ParamTree(SYNTH_CONFIG, seed=0).to(dev)
    eng = Engine(model)
    host = {k: v.pin_memory() for k, v in make_inputs(kind, B, T, seed=1 + rank).items()}
    inp = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
    src = inp.get("vc_src")

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- value: K graph-replayed iterations, inputs resident, CUDA events on the launch stream ----
    sess = eng.begin(kind, inp["vc_tgt"], inp["adv_tgt"], 0.1, W + K + 1, vc_src=src, w0=inp["w0"], want_loss=True)
    launches_per_iter = sess.launches_per_iter
    sess.step(W)
    prof = sess.profile()                                   # one eager iteration, events around every launch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    with ClockSampler(local) as clk:
        e0.record()
        sess.step(K)
        e1.record()
        barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    clocks = clk.summary()
    value = K * B * world / (ms / 1e3)
    adv, info = sess.end()                                  # the timed steps are the session's last iterations
    losses = info["losses"][: W + K + 1]
    if not bool(torch.isfinite(losses).all()):
        raise SystemExit("bench.py: non-finite loss")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"adv": adv, "losses": losses})

    # ---- roofline of the dominant kernel class (conv) from the per-launch event times ---------------
    peaks = load_peaks()
    by_kind = {}
    for k, t_ms, fl, by in prof:
        d = by_kind.setdefault(KIND_NAMES.get(k, str(k)), {"launches": 0, "ms": 0.0, "flops": 0.0, "bytes": 0.0})
        d["launches"] += 1; d["ms"] += t_ms; d["flops"] += fl; d["bytes"] += by
    tot_ms = sum(d["ms"] for d in by_kind.values()) or 1e-9
    conv = by_kind.get("conv", {"launches": 1, "ms": 1e-9, "flops": 0.0, "bytes": 0.0})
    # Per-launch event times of ~5 us kernels carry ~2 us of event overhead each, so the class SHARE comes
    # from the eager pass and the absolute time from the graph-replayed timed region.
    conv_share = conv["ms"] / tot_ms
    conv_ms_in_step = (ms / K) * conv_share
    conv_tf = conv["flops"] / (conv_ms_in_step / 1e3) / 1e12
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(f"{args.workload}_conv_dram_bytes_per_launch")
        except Exception:
            traffic = None
    roofline = {"bound": "tensor", "achieved": conv_tf, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                "frac": conv_tf / peaks["bf16_tflops"], "traffic": traffic,
                "kernel": "conv1d implicit GEMM (fwd + dgrad), all conv launches of one iteration"
                          + (" -- batch 1: latency-bound fp32 CUDA-core kernel conv_small_kernel, M <= 256 rows per GEMM" if B == 1 else ""),
                "launches": conv["launches"], "avg_launch_us": 1e3 * conv_ms_in_step / conv["launches"],
                "share_of_step": conv_share, "peak_source": peaks["source"] + ", bf16 dense burst",
                "algorithmic_gflop_per_launch": conv["flops"] / conv["launches"] / 1e9,
                "algorithmic_gflop_per_step": sum(d["flops"] for d in by_kind.values()) / 1e9}
    hbm = {}
    for name in ("norm", "update", "loss"):
        if name in by_kind and by_kind[name]["ms"] > 0:
            gbs = by_kind[name]["bytes"] / (by_kind[name]["ms"] / 1e3) / 1e9
            hbm[name] = {"achieved_gbs": gbs, "frac": gbs / peaks["hbm_gbs"], "launches": by_kind[name]["launches"],
                         "avg_launch_us": 1e3 * by_kind[name]["ms"] / by_kind[name]["launches"]}
    breakdown = {k: {"launches": d["launches"], "ms": round(d["ms"], 4)} for k, d in by_kind.items()}

    # ---- e2e: the drop-in public API with pinned host tensors ----------------------------------------
    fn = {"emb": AU.emb_attack, "e2e": AU.e2e_attack, "fb": AU.fb_attack}[kind]

    def public_call(n):
        d = {k: v.to(dev, non_blocking=True) for k, v in host.items() if k != "w0"}
        if kind == "emb":
            out = fn(model, d["vc_tgt"], d["adv_tgt"], 0.1, n)
        else:
            out = fn(model, d["vc_src"], d["vc_tgt"], d["adv_tgt"], 0.1, n)
        return out.cpu()
    public_call(3)
    barrier()
    t0 = time.perf_counter()
    res = public_call(K)
    torch.cuda.synchronize(dev)
    e2e_ms = max_over_ranks(1e3 * (time.perf_counter() - t0))
    e2e_value = K * B * world / (e2e_ms / 1e3)
    h2d = sum(v.numel() * 4 for k, v in host.items() if k != "w0")
    d2h = res.numel() * 4
    launches_before = eng.kernel_launches

    # ---- N > 1: the path that really shards -- BASELINE configs[3], emb_attack on 512 utterances of 80x512 per GPU
    # (4096 over 8) with the GLOBAL MSE normaliser, every rank holding only its own slice, and the one exchange step of
    # the workload (NCCL all_gather of the perturbed utterances + all_reduce of the loss curves) INSIDE the timed region.
    sharded = None
    if world > 1 and not args.no_extra:
        from attack_vc_b200.distributed import gather_shards, global_inv_norm
        Bs, Ts, ns = 512, 512, 6
        shard = {k: v.to(dev) for k, v in make_inputs("emb", Bs, Ts, seed=100 + rank).items()}
        inv = global_inv_norm("emb", Bs * world, 128, 80, Ts)
        s2 = eng.begin("emb", shard["vc_tgt"], shard["adv_tgt"], 0.1, 3 + ns, w0=shard["w0"], inv_norm=inv, want_loss=True)
        s2.step(3)
        ea, eb, ec = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        barrier()
        ea.record()
        s2.step(ns)
        eb.record()
        adv_l, inf2 = s2.end()
        adv_all, loss_all = gather_shards(adv_l, inf2["losses"], Bs * world)
        ec.record()
        barrier()
        ms_it = max_over_ranks(ea.elapsed_time(eb)) / ns
        ms_x = max_over_ranks(eb.elapsed_time(ec))
        sharded = {"workload": "BASELINE configs[3]: emb_attack, 80x512, 512 utterances per GPU, global 1/(B_total*128) normaliser",
                   "utterances_total": Bs * world, "iterations_timed": ns, "ms_per_iteration": ms_it,
                   "utterance_iterations_per_s": Bs * world * 1e3 / ms_it,
                   "exchange_ms": ms_x, "exchange": "finish kernels + NCCL all_gather_into_tensor of %.0f MB per rank + all_reduce of the loss curve" % (adv_l.numel() * 4 / 1e6),
                   "defended_utterances_per_s_at_1500_iters": Bs * world / ((1500 * ms_it + ms_x) / 1e3),
                   "gathered_shape": list(adv_all.shape), "loss_first_last": [float(loss_all[0]), float(loss_all[3 + ns - 1])],
                   "algorithmic_tflops": 2.0728e-3 * Bs * world / (ms_it / 1e3)}
        del shard, adv_all, adv_l

    line = {
        "metric": "attack iterations/s (x utterances)", "value": value, "unit": "utterance-iterations/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": desc, "attack": kind, "utterances_per_gpu": B, "frames": T, "eps": 0.1},
        "detail": {"defended_utterances_per_s_at_1500_iters": value / 1500.0,
                   "l2": "not flushed: iteration i+1 consumes iteration i's state and the 19.6 MB of weights stay hot by construction of the attack; the batched side measurements stream activations larger than L2",
                   "conv_impl": os.environ.get("AVC_CONV_IMPL", "auto"), "library": eng._lib.avc_version().decode()},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "utterance-iterations/s", "h2d_bytes_per_step": h2d / K, "d2h_bytes_per_step": d2h / K,
                "ms_total": e2e_ms, "api": f"attack_utils.{kind}_attack(model, ..., n_iters={K}) with pinned host tensors"},
        "gpu_launches": launches_per_iter * K,
        "launches_per_step": launches_per_iter,
        "roofline": roofline, "hbm_kernels": hbm, "breakdown_ms": breakdown, "sharded": sharded,
        "loss_first_last": [float(losses[0]), float(losses[-1])],
        "kernel_launches_total": launches_before,
    }

    # ---- side measurements on rank 0 at N=1: batched configs where the rooflines are meaningful ------
    if world == 1 and not args.no_extra and args.workload == "e2e":
        extra = {}
        for name, (k2, B2, T2, n2) in {"emb_B128_T512": ("emb", 128, 512, 6), "fb_B64_T256": ("fb", 64, 256, 6),
                                      "emb_B512_T512_cfg4_per_gpu": ("emb", 512, 512, 4)}.items():
            try:
                i2 = {k: v.to(dev) for k, v in make_inputs(k2, B2, T2, seed=9).items()}
                s2 = eng.begin(k2, i2["vc_tgt"], i2["adv_tgt"], 0.1, 3 + n2 + 1, vc_src=i2.get("vc_src"), w0=i2["w0"])
                s2.step(3)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize(dev)
                a.record(); s2.step(n2); b.record(); torch.cuda.synchronize(dev)
                ms2 = a.elapsed_time(b) / n2
                p2 = s2.profile(); s2.end()
                cf = sum(f for kk, _, f, _ in p2 if kk == 0); cm = sum(m for kk, m, _, _ in p2 if kk == 0)
                tf = cf / (cm / 1e3) / 1e12
                ent = {"utterance_iterations_per_s": B2 * 1e3 / ms2, "ms_per_step": ms2, "conv_tflops": tf,
                       "conv_frac_of_bf16_peak": tf / peaks["bf16_tflops"],
                       # tcgen05 path: per 8 input channels one TF32 MMA (hi*hi) and one BF16 K=16 MMA (lo*hi + hi*lo), each as long
                       # as a single-pass TF32 MMA: the tensor pipe executes 2x the algorithmic FLOPs at the TF32 rate (= bf16 peak / 2)
                       "conv_tensor_pipe_busy_frac": 2 * tf / (peaks["bf16_tflops"] / 2),
                       "conv_kernel": "conv_tc_kernel (tcgen05: kind::tf32 hi*hi + kind::f16 bf16 correction, chunked fp32 accumulation)",
                       "conv_share_of_step": cm / sum(m for _, m, _, _ in p2)}
                for kk, nm in ((1, "norm"), (5, "update")):
                    mm = sum(m for q, m, _, _ in p2 if q == kk); bb = sum(bt for q, _, _, bt in p2 if q == kk)
                    if mm > 0:
                        ent[nm + "_gbs"] = bb / (mm / 1e3) / 1e9
                        ent[nm + "_frac_of_hbm_peak"] = ent[nm + "_gbs"] / peaks["hbm_gbs"]
                extra[name] = ent
                del i2
            except Exception as e:   # a side measurement must never take the headline down
                extra[name] = {"error": str(e)[:200]}
        # HBM-bound kernels at a size where the HBM roofline applies (268 MB per tensor, >> L2), through the C-ABI unit
        # entry points, timed on the device over back-to-back launches.  SURVEY §8d bytes per element.
        try:
            Bn, Tn, Cn = 2048, 256, 128
            gen = torch.Generator(device="cpu").manual_seed(0)
            yn = torch.randn(Bn, Tn, Cn, generator=gen).to(dev); cn = torch.randn(Bn, 2 * Cn, generator=gen).to(dev)
            gn = torch.randn(Bn, Tn, Cn, generator=gen).to(dev)
            _, stn = eng.instnorm_adain_act_fwd(yn, cn, None, 1, 0.0)

            def med_ms(fn, reps=9):
                # device time per launch of `reps` launches back to back behind a first run (avc_unit_timing): a single
                # launch bracketed by events from Python carries ~20 us of host time between the first event and the launch
                eng.unit_timing(reps)
                try:
                    ts = []
                    for _ in range(3):
                        fn(); ts.append(eng.unit_last_ms())
                finally:
                    eng.unit_timing(0)
                return sorted(ts)[1]
            nel = Bn * Tn * Cn
            for nm, byt, fn in (("norm_fwd", 8, lambda: eng.instnorm_adain_act_fwd(yn, cn, None, 1, 0.0)),
                                ("norm_fwd_skip", 12, lambda: eng.instnorm_adain_act_fwd(yn, cn, gn, 1, 0.0)),
                                ("norm_bwd", 12, lambda: eng.instnorm_adain_act_bwd(gn, yn, stn, cn, 0.0))):
                msn = med_ms(fn)
                extra[f"{nm}_{Bn}x{Tn}x{Cn}"] = {"ms": msn, "gbs": byt * nel / msn / 1e6, "frac_of_hbm_peak": byt * nel / msn / 1e6 / peaks["hbm_gbs"],
                                                  "bytes_per_element": byt}
            del yn, cn, gn, stn
        except Exception as e:
            extra["norm_hbm_size"] = {"error": str(e)[:200]}
        line["batched"] = extra

    if world == 1 and not args.no_cpu_baseline:
        line["gpu_eager_baseline"] = gpu_eager_baseline(kind, min(B, 64), T, dev)
        Bc = min(B, 8)
        rate, cores, n, dt = cpu_loop_rate(kind, Bc, T, budget_s=15.0, max_iters=400)
        line["cpu_baseline"] = {"value": rate, "unit": "utterance-iterations/s", "cores": cores, "kind": "port",
                                "sample": f"{n} iterations of {kind}_attack, {Bc} utterance(s) of 80x{T}, oracle loop (bit-identical to the reference loop), {dt:.1f} s"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

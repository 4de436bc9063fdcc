"""Time per iteration of a ragged emb attack (Engine.attack_varlen, lengths uniform over 0.6-1.0 Tmax, the longest at Tmax)
against an equal-length Engine.attack at (B, Tmax), same engine, same command.  Per-iteration time = (t(400) - t(100)) / 300
with a host clock around calls that end in torch.cuda.synchronize(): plan building and setup cancel out.  The equal-length
call runs before and after the ragged one.  Dead rows of the padded layout should cost no more than live rows.

  python scripts/ragged_attack_timing.py
"""
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from attack_vc_b200 import Engine
from oracle import adainvc_oracle as O
eng = Engine(O.ParamTree(O.SYNTH_CONFIG, seed=0).to("cuda"))
def run(B, Tmax, ragged):
    g = torch.Generator().manual_seed(1)
    lens = sorted([int(t) for t in torch.randint(int(Tmax * 0.6), Tmax + 1, (B,), generator=g)], reverse=True) if ragged else [Tmax] * B
    lens[0] = Tmax
    mels = [torch.rand(T, 80, device="cuda") for T in lens]
    adv = torch.rand(1, 80, 128, device="cuda").expand(B, -1, -1)
    x = torch.rand(B, 80, Tmax, device="cuda")
    def once(n):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        if ragged: eng.attack_varlen("emb", mels, adv, 0.1, n)
        else: eng.attack("emb", x, adv, 0.1, n)
        torch.cuda.synchronize(); return time.perf_counter() - t0
    once(20); once(100)
    a, b = min(once(100) for _ in range(2)), min(once(400) for _ in range(2))
    return (b - a) / 300 * 1e3, sum(lens)
for B, Tmax in ((64, 320), (512, 640)):
    e, _ = run(B, Tmax, False); r, rows = run(B, Tmax, True); e2, _ = run(B, Tmax, False)
    print(f"B={B} Tmax={Tmax}: equal-length {e:.3f} / {e2:.3f} ms/iter, ragged (lengths 0.6-1.0 Tmax, {rows} of {B*Tmax} rows live) {r:.3f} ms/iter, ratio {r / min(e, e2):.3f}", flush=True)

"""Timing of the tower's tcgen05 GEMM alone at the bench workload's shapes, per epilogue (one box, interleaved A/B).

    python tools/ab_gemm.py [--rows 130000] [--acts 0]

Runs the four Linear layers of one ViT-H block (QKV, out-proj + residual, fc1 + activation, fc2 + residual) through
leaf_gemm_bf16 on random bf16 operands with M packed rows, alternating the activation codes given in --acts for the fc1
epilogue (0 = erf GELU, 1 = QuickGELU) so that clock drift hits all of them alike. Prints
microseconds per launch and TFLOP/s; the operands (> 1 GB per launch) are far larger than L2, so no flush is needed.
"""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from leaf_b200 import synth                                  # noqa: E402
from leaf_b200.tower import LeafTextTower                    # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=130000)
    ap.add_argument("--acts", type=int, nargs="+", default=[0])
    ap.add_argument("--reps", type=int, default=6)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    W, M = 1024, a.rows
    eng = LeafTextTower.random(synth.TowerCfg("ab", W, 1, 16, 1024), seed=0, device=dev).leaf_engine
    g = torch.Generator(device=dev).manual_seed(0)
    rnd = lambda *s: (torch.randn(s, device=dev, generator=g) * 0.5)
    A1 = rnd(M, W).to(torch.bfloat16)
    A4 = rnd(M, 4 * W).to(torch.bfloat16)
    x = rnd(M, W)
    Wq, Wo, W1, W2 = (rnd(3 * W, W) * 0.06).to(torch.bfloat16), (rnd(W, W) * 0.06).to(torch.bfloat16), \
        (rnd(4 * W, W) * 0.06).to(torch.bfloat16), (rnd(W, 4 * W) * 0.03).to(torch.bfloat16)
    bq, bo, b1, b2 = rnd(3 * W), rnd(W), rnd(4 * W), rnd(W)
    Cq = torch.empty((M, 3 * W), dtype=torch.bfloat16, device=dev)
    C1 = torch.empty((M, 4 * W), dtype=torch.bfloat16, device=dev)
    cases = [("qkv  (bf16 store)", lambda: eng.gemm(A1, Wq, bq, 0, 0, Cq), 6)]
    for act in a.acts:
        cases.append((f"fc1  (act code {act})", (lambda act=act: eng.gemm(A1, W1, b1, 1, act, C1)), 8))
    Co = torch.empty((M, W), dtype=torch.bfloat16, device=dev)
    cases += [("out  (fp32 residual)", lambda: eng.gemm(A1, Wo, bo, 2, 0, x), 2),
              ("out  (bf16 store)", lambda: eng.gemm(A1, Wo, bo, 0, 0, Co), 2),
              ("fc2  (fp32 residual)", lambda: eng.gemm(A4, W2, b2, 2, 0, x), 8)]
    if len(a.acts) > 1:                                       # the activation variants must agree to bf16 rounding
        ref = eng.gemm(A1, W1, b1, 1, a.acts[0]).float()
        for act in a.acts[1:]:
            d = (eng.gemm(A1, W1, b1, 1, act).float() - ref).abs()
            print(f"act {act} vs act {a.acts[0]}: max |diff| {d.max().item():.3g}, differing elements {(d > 0).float().mean().item():.2%}")
    times = {name: [] for name, _, _ in cases}
    for rep in range(a.reps):
        for name, fn, _ in cases:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(8):
                fn()
            e1.record()
            torch.cuda.synchronize()
            if rep:
                times[name].append(e0.elapsed_time(e1) / 8)
    for name, _, units in cases:
        ms = sum(times[name]) / len(times[name])
        print(f"{name:24s} {ms * 1e3:8.1f} us   {M * units * W * W / ms / 1e9:7.1f} TFLOP/s")


if __name__ == "__main__":
    main()

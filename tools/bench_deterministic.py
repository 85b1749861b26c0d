"""What deterministic mode (torch.use_deterministic_algorithms(True) -> leaf_set_deterministic) costs.

At bench.py's K4 shape (B clean captions standing in for the winners, random-init tower of the named shape) it times, with CUDA
events on the launching stream and the two modes interleaved iteration by iteration:
  * leaf_forward_train + loss + leaf_backward (K4) for every tower of --towers;
  * one whole FareTrainer.step (anchors, attack, K4, AdamW) on the first tower.
On the first tower it also takes one torch.profiler pass per mode (a separate run, after the timed ones) and lists the kernels
whose total time differs most between the modes. Prints one JSON line with the GPU's name and power limit read in the same run.

    python tools/bench_deterministic.py --towers ViT-H-14,ViT-L-14,ViT-bigG-14 --iters 30
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"nvidia-smi failed: {q.stderr.strip()}"


def summary(xs):
    xs = sorted(xs)
    return dict(median_ms=statistics.median(xs), min_ms=xs[0], max_ms=xs[-1], n=len(xs))


def k4_once(tower, tok, lens, anchor):
    tower.zero_grad()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    f = tower.encode_text(tok, host_lengths=lens)
    torch.nn.functional.mse_loss(anchor, f, reduction="none").sum(dim=-1).mean().backward()
    b.record()
    return a, b


def time_k4(name, B, iters, warmup):
    from leaf_b200 import synth
    from leaf_b200.tower import LeafTextTower
    cfg = synth.TOWERS[name]
    tower = LeafTextTower.random(name, seed=0).trainable()
    caps = synth.make_captions(B, seed=1)
    tok, lens = tower.tokenizer(caps, with_lengths=True)
    anchor = torch.randn((B, cfg.embed_dim), generator=torch.Generator(device="cuda").manual_seed(2), device="cuda")
    ev = {False: [], True: []}
    for i in range(warmup + iters):
        for det in (False, True):
            torch.use_deterministic_algorithms(det)
            e = k4_once(tower, tok, lens, anchor)
            if i >= warmup:
                ev[det].append(e)
    torch.cuda.synchronize()
    torch.use_deterministic_algorithms(False)
    ms = {det: [a.elapsed_time(b) for a, b in v] for det, v in ev.items()}
    out = dict(packed_rows=int(sum(lens)), sequences=B, default=summary(ms[False]), deterministic=summary(ms[True]))
    out["ratio_of_medians"] = out["deterministic"]["median_ms"] / out["default"]["median_ms"]
    return out, (tower, tok, lens, anchor)


def profile_k4(state, top=12):
    """Per-kernel CUDA time of one K4 iteration per mode (torch.profiler, its own pass): the kernels whose totals differ most."""
    from torch.profiler import ProfilerActivity, profile
    tower, tok, lens, anchor = state
    per = {}
    for det in (False, True):
        torch.use_deterministic_algorithms(det)
        k4_once(tower, tok, lens, anchor)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            k4_once(tower, tok, lens, anchor)
            torch.cuda.synchronize()
        per[det] = {e.key: (getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) / 1e3, e.count) for e in prof.key_averages()}
    torch.use_deterministic_algorithms(False)
    keys = set(per[False]) | set(per[True])
    rows = []
    for k in keys:
        d0, n0 = per[False].get(k, (0.0, 0))
        d1, n1 = per[True].get(k, (0.0, 0))
        rows.append(dict(kernel=k[:120], default_ms=round(d0, 4), default_launches=n0, deterministic_ms=round(d1, 4), deterministic_launches=n1,
                         delta_ms=round(d1 - d0, 4)))
    rows.sort(key=lambda r: -abs(r["delta_ms"]))
    return dict(total_default_ms=round(sum(v[0] for v in per[False].values()), 3),
                total_deterministic_ms=round(sum(v[0] for v in per[True].values()), 3), largest_differences=rows[:top])


def time_train_step(name, B, steps, rho):
    from leaf_b200 import synth
    from leaf_b200.fare import FareTrainer
    from leaf_b200.tower import LeafTextTower
    cfg = synth.TOWERS[name]
    sd = synth.random_tower_state_dict(cfg, seed=0, device="cuda")
    frozen = LeafTextTower(synth.perturbed_copy(sd, seed=1, std=1e-3), heads=cfg.heads)
    tr = FareTrainer(LeafTextTower(sd, heads=cfg.heads), frozen, rho=rho, k_adv=1, accum_freq=1, grad_clip_norm=1.0, lr=1e-5)
    ms = {False: [], True: []}
    for i in range(1 + steps):
        for det in (False, True):
            torch.use_deterministic_algorithms(det)
            np.random.seed(i)
            texts = synth.make_captions(B, seed=100 + i)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            tr.step(texts)
            b.record()
            torch.cuda.synchronize()
            if i >= 1:
                ms[det].append(a.elapsed_time(b))
    torch.use_deterministic_algorithms(False)
    out = dict(sequences=B, rho=rho, default=summary(ms[False]), deterministic=summary(ms[True]))
    out["ratio_of_medians"] = out["deterministic"]["median_ms"] / out["default"]["median_ms"]
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--towers", default="ViT-H-14,ViT-L-14,ViT-bigG-14")
    ap.add_argument("--B", type=int, default=128)
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--train-steps", type=int, default=5)
    ap.add_argument("--rho", type=int, default=50)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_deterministic: no CUDA device (the engine has no CPU path)")
    towers = a.towers.split(",")
    line = dict(gpu=gpu_info(), torch=torch.__version__, B=a.B, iters=a.iters, k4={})
    prof = None
    for i, name in enumerate(towers):
        line["k4"][name], state = time_k4(name, a.B, a.iters, a.warmup)
        if i == 0:
            prof = profile_k4(state)
        del state
        torch.cuda.empty_cache()
    line["k4_profile_" + towers[0]] = prof
    if a.train_steps > 0:
        line["fare_step_" + towers[0]] = time_train_step(towers[0], a.B, a.train_steps, a.rho)
    line["gpu_after"] = gpu_info()
    print(json.dumps(line))


if __name__ == "__main__":
    main()

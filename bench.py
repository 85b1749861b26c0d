#!/usr/bin/env python
"""LEAF candidates scored per second (BASELINE.json metric).

    python bench.py [--gpus N --steps K --warmup W]            # this repo's engine on N B200s (torchrun for N > 1)
    python bench.py --impl reference [--steps K --warmup W]    # the reference algorithm on the host CPU (oracle port)
    python bench.py --dump-outputs DIR ...                     # also write the last timed step's results to DIR/*.npy

One "step" = one attack_text_leaf call on one batch of synthetic captions: 2*k*B*rho candidates expanded, tokenized,
encoded by the text tower and scored (SURVEY.md 8d). Prints ONE JSON line on rank 0.
  value : device-resident throughput (captions and draws already in HBM, CUDA events around the kernels)
  e2e   : the same through leaf_b200.attack_text_leaf with host strings (H2D of captions/draws and D2H of the
          winners inside the timed region)
The inputs (tower weights, captions, draws, anchors) are seeded and computed without this repo's kernels, so two builds
run with the same arguments can be compared output for output with --dump-outputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import zlib

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from leaf_b200 import synth  # noqa: E402

METRIC = "leaf_candidates_scored_per_sec"
UNIT = "candidates/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="ViT-H-14")
    ap.add_argument("--batch", type=int, default=128, help="captions per GPU per step")
    ap.add_argument("--rho", type=int, default=50)
    ap.add_argument("--k", type=int, default=1)
    ap.add_argument("--captions", default="typical", choices=["typical", "dense-77", "short"])
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train-step", action="store_true", help="skip the full FARE step (attack + K4 + AdamW) leg")
    ap.add_argument("--no-overlap-allreduce", action="store_true", help="FARE step: one blocking all-reduce after the backward instead of the per-layer overlapped exchange")
    ap.add_argument("--no-library-baseline", action="store_true", help="skip the stock-PyTorch-on-the-same-GPU leg (N = 1 only)")
    ap.add_argument("--no-dense77", action="store_true", help="skip the worst-case (every row truncated to 77 tokens) leg")
    ap.add_argument("--no-global-batch", action="store_true", help="skip the strong-scaling legs with a collective on the path (N > 1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed on rank 0 "
                    "(winning position and character index per caption, winner features) as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def dump_outputs(path, arrays, limit=DUMP_LIMIT_BYTES, seed=0):
    """Writes `arrays` (name -> array, one row per caption) as path/<name>.npy, floats as float32 / float64 and integers as
    float64 (exact). When they hold more than `limit` bytes, the same seeded sample of rows is written for every array, with
    the sampled row indices as path/rows.npy."""
    os.makedirs(path, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, dtype=np.float32 if v.dtype == np.float32 else np.float64) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = sum(v.nbytes for v in arrays.values()) // max(n, 1) + 8
    if n * row_bytes > limit:
        rows = np.sort(np.random.RandomState(seed).choice(n, size=limit // row_bytes, replace=False))
        arrays = {k: v[rows] for k, v in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), v)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1415.6), d.get("hbm_gbs", 6452.2), "measured (MEASURED_PEAKS.json, sustained bf16)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


def workload_name(a):
    return f"{a.model} text tower, LEAF k={a.k} rho={a.rho}, batch {a.batch} {a.captions} synthetic captions per GPU"


# ------------------------------------------------------------------------------------------------------------------
# CPU reference arm / cpu_baseline: the oracle port of attack_text_leaf on the host cores
# ------------------------------------------------------------------------------------------------------------------
def cpu_attack_rate(a, seconds, steps=1, warmup=0):
    """Times oracle.attack_text_leaf_oracle (fp32 torch CPU, all host threads) on a bounded sample of the workload:
    same tower shape, same caption generator, same rho and k, reduced batch so that one call fits `seconds`."""
    from oracle import leaf_oracle as O
    cfg = synth.TOWERS[a.model]
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    sd = synth.random_tower_state_dict(cfg, seed=0)
    frozen = synth.perturbed_copy(sd, seed=1, std=1e-3)
    otok = O.OracleTokenizer()
    enc = lambda t, normalize: O.encode_text(sd, t, cfg.heads, quick_gelu=cfg.quick_gelu, normalize=normalize)
    # calibrate: one 77-slot row batch to estimate seconds per candidate
    caps = synth.make_captions(max(a.batch, 4), seed=0, kind=a.captions)
    with torch.no_grad():
        t0 = time.perf_counter()
        enc(otok(caps[:2] * 4), False)
        per_cand = (time.perf_counter() - t0) / 8
    per_call_budget = seconds / max(steps + warmup, 1)
    B = int(max(1, min(a.batch, per_call_budget / (per_cand * 2 * a.k * a.rho))))
    caps = caps[:B]
    times = []
    with torch.no_grad():
        anchor = O.encode_text(frozen, otok(caps), cfg.heads, quick_gelu=cfg.quick_gelu)
        for it in range(warmup + steps):
            np.random.seed(it)
            t0 = time.perf_counter()
            O.attack_text_leaf_oracle(enc, otok, caps, anchor, objective="l2", n=a.rho, k=a.k)
            dt = time.perf_counter() - t0
            if it >= warmup:
                times.append(dt)
    cands = 2 * a.k * B * a.rho
    ms = 1e3 * sum(times) / len(times)
    return dict(value=cands / (ms / 1e3), unit=UNIT, cores=threads, kind="port",
                sample=f"oracle port of attack_text_leaf (fp32 torch CPU, dense 77-slot rows as the reference computes), "
                       f"{a.model}, B={B} of {a.batch}, rho={a.rho}, k={a.k}, {a.captions} captions, {len(times)} call(s)",
                extrapolation=f"candidates/s measured on {cands} candidates per call; the reference encodes every candidate as its own "
                              f"dense 77-slot row, so its cost is linear in the candidate count and the rate carries over to the "
                              f"{2 * a.k * a.batch * a.rho}-candidate step unchanged (full step ~ {2 * a.k * a.batch * a.rho / (cands / (ms / 1e3)):.0f} s on these cores)"), ms, cands


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    base, ms, cands = cpu_attack_rate(a, seconds=120.0, steps=a.steps, warmup=min(a.warmup, 1))
    line = dict(metric=METRIC, value=base["value"], unit=UNIT, n_gpus=a.gpus, steps=a.steps, warmup=a.warmup, ms_per_step=ms,
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic", impl="reference",
                config=dict(workload=workload_name(a), candidates_per_step=cands), cpu_baseline=base,
                e2e=dict(value=base["value"], unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# GPU library baseline: the reference's stock PyTorch path on the SAME B200 (SURVEY.md 8d, last bullet)
# ------------------------------------------------------------------------------------------------------------------
def _torch_tower(sd, tok, heads, quick):
    """CLIP.encode_text (model.py:269-284) as the ATen / cuBLAS / SDPA kernels the reference's modules launch: F.layer_norm,
    nn.Linear, nn.MultiheadAttention's fused scaled_dot_product_attention path (need_weights=False), nn.GELU, dense 77-slot
    rows - none of this repo's kernels."""
    F = torch.nn.functional
    N, T = tok.shape
    x = sd["token_embedding.weight"][tok] + sd["positional_embedding"][:T]
    W = x.shape[-1]
    d = W // heads
    i = 0
    while f"transformer.resblocks.{i}.ln_1.weight" in sd:
        p = f"transformer.resblocks.{i}."
        h = F.layer_norm(x, (W,), sd[p + "ln_1.weight"], sd[p + "ln_1.bias"], 1e-5)
        qkv = F.linear(h, sd[p + "attn.in_proj_weight"], sd[p + "attn.in_proj_bias"])
        q, k, v = (z.view(N, T, heads, d).transpose(1, 2) for z in qkv.split(W, dim=-1))
        o = F.scaled_dot_product_attention(q, k, v, is_causal=True).transpose(1, 2).reshape(N, T, W)
        x = x + F.linear(o, sd[p + "attn.out_proj.weight"], sd[p + "attn.out_proj.bias"])
        h = F.layer_norm(x, (W,), sd[p + "ln_2.weight"], sd[p + "ln_2.bias"], 1e-5)
        h = F.linear(h, sd[p + "mlp.c_fc.weight"], sd[p + "mlp.c_fc.bias"])
        h = h * torch.sigmoid(1.702 * h) if quick else F.gelu(h)
        x = x + F.linear(h, sd[p + "mlp.c_proj.weight"], sd[p + "mlp.c_proj.bias"])
        i += 1
    x = F.layer_norm(x, (W,), sd["ln_final.weight"], sd["ln_final.bias"], 1e-5)
    return x[torch.arange(N, device=x.device), tok.argmax(dim=-1)].float() @ sd["text_projection"]


def gpu_library_baseline(a, sd, caps, anchor, cfg, dev):
    """attack_text_leaf as the reference runs it on a GPU (utils_attacks.py:297-393 via the oracle's restatement of the loop):
    candidate strings and SimpleTokenizer on the HOST, every candidate a dense 77-slot row, the tower in stock PyTorch on
    the same B200 - (i) as shipped: fp32 weights, TF32 matmuls (train_AT_text_only.py:99), no autocast; (ii) under
    torch.autocast(bfloat16) for a like-for-like precision comparison. One timed call each after a small warm-up call; host
    tokenization time is reported separately from device time."""
    from oracle import leaf_oracle as O
    otok = O.OracleTokenizer()
    out = {}
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    try:
        for name in ("fp32_tf32", "bf16_autocast"):
            torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = True
            host_s, dev_ms = [0.0], [0.0]

            def tokenize(texts):
                t0 = time.perf_counter()
                t = otok(texts)
                host_s[0] += time.perf_counter() - t0
                return t

            def encode(tok, normalize):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                with torch.autocast("cuda", dtype=torch.bfloat16, enabled=(name == "bf16_autocast")):
                    f = _torch_tower(sd, tok.to(dev), cfg.heads, cfg.quick_gelu)
                f = torch.nn.functional.normalize(f, dim=-1) if normalize else f
                e1.record()
                e1.synchronize()
                dev_ms[0] += e0.elapsed_time(e1)
                return f

            with torch.no_grad():
                np.random.seed(1)
                O.attack_text_leaf_oracle(encode, tokenize, caps[:4], anchor[:4].clone(), objective="l2", n=a.rho, k=a.k)   # warm-up
                host_s[0] = dev_ms[0] = 0.0
                np.random.seed(2000)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                O.attack_text_leaf_oracle(encode, tokenize, caps, anchor.clone(), objective="l2", n=a.rho, k=a.k)
                torch.cuda.synchronize()
                wall = time.perf_counter() - t0
            cands = 2 * a.k * len(caps) * a.rho
            out[name] = dict(e2e_candidates_per_s=cands / wall, device_candidates_per_s=cands / (dev_ms[0] * 1e-3), wall_ms=wall * 1e3,
                             device_ms=dev_ms[0], host_tokenize_ms=host_s[0] * 1e3,
                             dense77_tflops=cands * cfg.dense_flops_per_candidate / (dev_ms[0] * 1e-3) / 1e12)
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    out["what"] = ("the reference's attack loop with its stock PyTorch tower on this GPU: host candidate strings + host BPE "
                   "(oracle tokenizer, pure Python like SimpleTokenizer), dense 77-slot rows, ATen/cuBLAS/SDPA kernels; "
                   f"B={len(caps)}, rho={a.rho}, k={a.k}, one call")
    return out


# ------------------------------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------------------------------
class Clocks:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.samples, self.stop = index, [], threading.Event()
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *exc):
        self.stop.set()
        self.t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["unavailable"])
        mhz = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(s) > 2 + i and s[2 + i].lower().startswith("active") for s in self.samples)]
        mx = [int(s[1]) for s in self.samples if s[1].isdigit()]
        return dict(sm_mhz=mhz[len(mhz) // 2] if mhz else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons,
                    samples=len(self.samples))


# ------------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------------
def run_ours(a):
    import torch.distributed as dist
    from leaf_b200 import attack_text_leaf
    from leaf_b200.attack import V_DEFAULT
    from leaf_b200.tower import LeafTextTower
    from oracle import leaf_oracle as O

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = synth.TOWERS[a.model]
    B, n, k = a.batch, a.rho, a.k
    # the path shards by samples: every rank attacks its own batch, no collective on the data path (weak scaling)
    tower = LeafTextTower.random(a.model, seed=0, device=dev)
    eng = tower.leaf_engine
    caps = synth.make_captions(B, seed=100 + rank, kind=a.captions)
    frozen_sd = synth.perturbed_copy(tower.open_clip_state_dict(), seed=1, std=1e-3)
    otok = O.OracleTokenizer()

    def frozen_anchor(cs):
        """E_frozen(x) by the fp32 oracle tower on this GPU, not by this repo's kernels: the anchors are the same whichever
        build is measured."""
        tok = otok(cs).to(dev)
        with torch.no_grad():
            return torch.cat([O.encode_text_device(frozen_sd, tok[s:s + 256], cfg.heads, quick_gelu=cfg.quick_gelu)
                              for s in range(0, len(cs), 256)])

    anchor = frozen_anchor(caps)
    dense_caps = synth.make_captions(B, seed=100 + rank, kind="dense-77")
    dense_anchor = frozen_anchor(dense_caps)
    gcaps = synth.make_captions(B, seed=100, kind=a.captions)               # ONE global batch, identical on every rank
    ganchor = frozen_anchor(gcaps)
    del frozen_sd
    torch.cuda.empty_cache()
    eng.reserve(B * n + B)
    Vt = np.asarray(V_DEFAULT, dtype=np.int32)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)      # > 126 MB L2

    def draws(seed, cs=None):
        cs = caps if cs is None else cs
        rs = np.random.RandomState(seed)
        pos = np.stack([rs.choice(range(2 * len(S) + 1), size=n, replace=n > 2 * len(S) + 1) for S in cs]).astype(np.int32)
        ch = Vt[np.stack([rs.choice(range(len(Vt)), size=n, replace=n > len(Vt)) for _ in cs])]
        return torch.from_numpy(pos).to(dev), torch.from_numpy(ch).to(dev)

    typical_set = eng.upload_captions(caps) + (anchor,)
    space = torch.full((B * n,), 32, dtype=torch.int32, device=dev)

    def device_step(pos_d, chr_d, record=None, cset=None):
        """The hot path with inputs resident in HBM (k = 1 form: no host round trip between the phases). Returns the
        winning position index [B], the winning character index [B] and the winner's features [B, E]."""
        caps_d, off_d, anc = typical_set if cset is None else cset
        tok, ln, base = eng.expand_tokenize(caps_d, off_d, B, n, pos=pos_d, chr_=space)
        f = eng.encode_tokens(tok, ln, False, base, (B * n, n), trim=True)
        if record is not None:
            record.append((ln[:B * n], eng.last_rows()))
        best1, _, _ = eng.score(f, anc, B, n, "l2")
        tok, ln, base = eng.expand_tokenize(caps_d, off_d, B, n, pos=pos_d, chr_=chr_d, sel=best1)
        f = eng.encode_tokens(tok, ln, False, base, (B * n, n), trim=True)
        if record is not None:
            record.append((ln[:B * n], eng.last_rows()))
        best2, best_feat, _ = eng.score(f, anc, B, n, "l2")
        return best1, best2, best_feat

    def barrier():
        if world > 1:
            dist.barrier()

    # ---- device-resident timing ----
    all_draws = [draws(s) for s in range(a.warmup + a.steps)]
    for i in range(a.warmup):
        device_step(*all_draws[i])
    torch.cuda.synchronize()
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    lens_rec = []
    eng.launch_count(reset=True)
    with Clocks(local) as clk:
        torch.cuda.synchronize()
        for i in range(a.steps):
            flush.fill_(i)                                  # L2 flush between timed iterations (outside the events)
            ev[i][0].record()
            for _ in range(k):
                last = device_step(*all_draws[a.warmup + i])
            ev[i][1].record()
        torch.cuda.synchronize()
        launches = eng.launch_count()
        if a.dump_outputs and rank == 0:
            dump_outputs(a.dump_outputs, dict(zip(("best_position", "best_character", "best_features"), (t.cpu().numpy() for t in last))))
        barrier()
        dev_ms = sum(s.elapsed_time(e) for s, e in ev)
        # ---- end to end through the public API (host strings in, winners out) ----
        for i in range(min(a.warmup, 2)):
            np.random.seed(1000 + i)
            attack_text_leaf(tower, None, caps, anchor.clone(), dev, objective="l2", n=n, k=k)
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        for i in range(a.steps):
            np.random.seed(2000 + i)
            feats, adv = attack_text_leaf(tower, None, caps, anchor.clone(), dev, objective="l2", n=n, k=k)
            float(feats[0, 0].item())                       # device -> host read of the step's result
        torch.cuda.synchronize()
        e2e_ms = (time.perf_counter() - t0) * 1e3
        barrier()
        # ---- the same with the reference's --constrain filter (every shipped training script enables it), masks computed
        #      on the device against a synthetic word list; the headline stays the unconstrained attack ----
        eng.load_words(synth.word_list(100 + rank))
        np.random.seed(1500)
        attack_text_leaf(tower, None, caps, anchor.clone(), dev, objective="l2", n=n, k=k, constrain=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(a.steps):
            np.random.seed(2000 + i)
            feats, adv_c = attack_text_leaf(tower, None, caps, anchor.clone(), dev, objective="l2", n=n, k=k, constrain=True)
            float(feats[0, 0].item())
        torch.cuda.synchronize()
        con_ms = (time.perf_counter() - t0) * 1e3
        changed = sum(x != y for x, y in zip(adv_c, caps))
        barrier()
    dev_ms_local, e2e_ms_local = dev_ms, e2e_ms
    t = torch.tensor([dev_ms, e2e_ms, con_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, con_ms = t.tolist()
    cands_step = 2 * k * B * n
    total_cands = cands_step * a.steps * world

    # ---- the whole FARE training step (utils_AT.py:291-366): attack + winners' forward/backward (K4) + data-parallel
    #      gradient all-reduce (NCCL) + AdamW + refresh of the engine's bf16 operand copies. Reported next to the
    #      headline; the headline metric stays "candidates scored per second" of the attack itself. ----
    train = None
    if not a.no_train_step:
        from leaf_b200.fare import FareTrainer
        frozen2 = LeafTextTower(synth.perturbed_copy(tower.open_clip_state_dict(), seed=1, std=1e-3), heads=cfg.heads,
                                quick_gelu=cfg.quick_gelu, device=dev)
        trainer = FareTrainer(tower, frozen2, rho=n, k_adv=k, lr=1e-5, wd=1e-4, beta1=0.9, beta2=0.98, eps=1e-6,   # scripts/train_leaf_vith.sh
                              overlap_allreduce=not a.no_overlap_allreduce)

        def train_step(seed):
            np.random.seed(seed)
            loss, _ = trainer.step(caps)
            return float(loss.item())

        train_step(3000)
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        losses = [train_step(3001 + i) for i in range(a.steps)]
        torch.cuda.synchronize()
        tr_ms = (time.perf_counter() - t0) * 1e3 / a.steps
        tt = torch.tensor([tr_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        train = dict(ms_per_step=tt.item(), attack_ms_per_step=e2e_ms / a.steps, loss_first=losses[0], loss_last=losses[-1],
                     what="leaf_b200.fare.FareTrainer.step: frozen anchors + attack_text_leaf + tokenize winners + forward/backward "
                          "(K4, gradients accumulated into one flat buffer) + " + (("NCCL all-reduce (" + ("one blocking call after the backward" if a.no_overlap_allreduce else "per-layer slices on a side stream while the backward runs") + ") + ") if world > 1 else "")
                          + "native AdamW (one launch) + weight refresh")
        tower.trainable(False)
        del trainer, frozen2

    # ---- K4 alone: forward (activations kept) + backward of B winners, CUDA events, with its own roofline entry ----
    W, L, E = cfg.width, cfg.layers, cfg.embed_dim
    peak_tf, peak_gbs, peak_src = peaks()
    k4 = None
    if not a.no_train_step:
        tok_w = tower.tokenizer(caps)
        rows_w = int((tok_w.argmax(dim=-1) + 1).sum().item())
        tower.trainable(True)
        tower.attach_grads()
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(a.steps)]
        for i in range(2 + a.steps):
            tower.zero_grad()
            if i >= 2:
                evs[i - 2][0].record()
            f = tower.encode_text(tok_w)
            if i >= 2:
                evs[i - 2][1].record()
            torch.nn.functional.mse_loss(anchor, f, reduction="none").sum(dim=-1).mean().backward()
            if i >= 2:
                evs[i - 2][2].record()
        torch.cuda.synchronize()
        fwd_ms = sum(e[0].elapsed_time(e[1]) for e in evs) / a.steps
        bwd_ms = sum(e[1].elapsed_time(e[2]) for e in evs) / a.steps
        k4_flops = 3.0 * (24.0 * W * W * rows_w * L + 2.0 * W * E * B)           # forward + data gradients + weight gradients
        k4_tf = k4_flops / ((fwd_ms + bwd_ms) * 1e-3) / 1e12
        k4 = dict(bound="tensor", achieved=k4_tf, peak=peak_tf, unit="TFLOP/s", frac=k4_tf / peak_tf, forward_ms=fwd_ms, backward_ms=bwd_ms,
                  packed_rows=rows_w, sequences=B, executed_gemm_tflop=k4_flops / 1e12,
                  what="leaf_forward_train + loss + leaf_backward of the B clean captions (stand-ins for the winners), CUDA events on the "
                       "launching stream; FLOPs = 3 x (24 W^2 rows L + 2 W E B)")
        tower.zero_grad()
        tower.trainable(False)

    # ---- roofline of the dominant kernel (the tcgen05 GEMM): extra steps with CUDA events around every GEMM launch ----
    def gemm_roofline(step_draws, cset, steps):
        rec = []
        device_step(*step_draws, record=rec, cset=cset)      # row counts (synchronises) + warm-up after the legs above
        torch.cuda.synchronize()
        eng.set_timing(True)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tot = 0.0
        for i in range(steps):                               # averaged over `steps` steps
            flush.fill_(i)
            ev0.record()
            device_step(*step_draws, cset=cset)              # the draws whose row counts were recorded above
            ev1.record()
            ev1.synchronize()
            tot += ev0.elapsed_time(ev1)
        per_step = lambda t: (t[0] / steps, t[1] // steps)
        gemm_ms, gemm_launches = per_step(eng.gemm_time_ms())
        insitu = {name: round(per_step(eng.class_time_ms(i))[0], 3) for i, name in enumerate(("gemm", "layernorm", "attention", "pack_embed"))}
        for epi, name in enumerate(("gemm_qkv_bf16", "gemm_fc1_bf16_act", "gemm_out_fc2_residual", "gemm_proj_f32", "gemm_fc2_residual", "gemm_out_bf16")):
            ms_epi, n_epi = per_step(eng.class_time_ms(4 + epi))
            if n_epi:
                insitu[name] = [round(ms_epi, 3), n_epi]
        eng.set_timing(False)
        lens = torch.cat([r[0] for r in rec]).double().cpu().numpy()
        rows_exec = sum(r[1] for r in rec)                                    # packed rows the GEMMs really processed
        # executed by the GEMM launches: every packed row through L-1 whole layers and the final layer's QKV projection; the
        # final layer's out-proj + MLP and the text projection see one (pooled EOS) row per sequence
        seqs = len(rec) * (B * n + B)
        gemm_flops = rows_exec * ((L - 1) * 24.0 + 6.0) * W * W + seqs * (18.0 * W * W + 2.0 * W * E)
        return dict(gemm_ms=gemm_ms, gemm_launches=gemm_launches, insitu=insitu, lens=lens, rows_exec=rows_exec, gemm_flops=gemm_flops,
                    step_ms_timed=tot / steps)

    r = gemm_roofline(all_draws[-1], None, a.steps)
    gemm_ms, gemm_launches, insitu, lens, rows_exec, gemm_flops = (r[k] for k in ("gemm_ms", "gemm_launches", "insitu", "lens", "rows_exec", "gemm_flops"))
    gemm_flops_credit = float((L * 24.0 * lens * W * W + 2.0 * W * E).sum())   # GEMM share of F(t), SURVEY.md 8d
    alg_flops = float(sum(cfg.flops_for_length(int(x)) for x in lens))
    achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    step_ms = dev_ms / a.steps
    traffic = None                                  # DRAM bytes per GEMM launch from the committed ncu --set full capture
    tp = os.path.join(ROOT, "profiles", "gemm_traffic.json")
    if os.path.exists(tp):
        tj = json.load(open(tp))
        if tj.get("workload") == workload_name(a):
            traffic = tj["dram_bytes_per_launch"]
    # HBM-bound companions of the GEMM, same in-situ events: algorithmic bytes per packed row and layer (DESIGN.md section 4)
    rows_layers = rows_exec * (L - 1) + rows_exec                               # attention and ln_1 run on every layer's packed rows
    att_gbs = 8.0 * W * rows_layers / (insitu["attention"] * 1e-3) / 1e9 if insitu.get("attention") else None
    ln_bytes = (6.0 * W * rows_exec * L + 8.0 * W * rows_exec * (L - 1))         # ln_1 every layer, ln_2 (+ bf16 delta) on the L-1 full layers
    ln_gbs = ln_bytes / (insitu["layernorm"] * 1e-3) / 1e9 if insitu.get("layernorm") else None
    roofline = dict(bound="tensor", achieved=achieved, peak=peak_tf, unit="TFLOP/s", frac=achieved / peak_tf, traffic=traffic,
                    kernel="gemm2_bf16_tn_kernel (tcgen05.mma.cta_group::2, all four Linear layers + projection)", peak_source=peak_src, gemm_launches_per_step=gemm_launches,
                    gemm_ms_per_step=gemm_ms, gemm_share_of_step=gemm_ms / step_ms if step_ms else None,
                    in_situ_ms_per_step=insitu,
                    algorithmic_tflop_per_step=alg_flops / 1e12, executed_gemm_tflop_per_step=gemm_flops / 1e12,
                    credited_gemm_tflops=gemm_flops_credit / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else None,
                    rows_executed_per_step=int(rows_exec), rows_without_prefix_sharing=int(lens.sum()),
                    whole_step_tflops=alg_flops / (step_ms * 1e-3) / 1e12 if step_ms else None,
                    whole_step_executed_frac=gemm_flops / (step_ms * 1e-3) / 1e12 / peak_tf if step_ms else None,
                    dense77_equiv_tflops=cands_step * cfg.dense_flops_per_candidate / (step_ms * 1e-3) / 1e12 if step_ms else None,
                    mean_len=float(lens.mean()),
                    hbm_kernels=dict(peak_gbs=peak_gbs,
                                     attention=dict(achieved_gbs=att_gbs, frac=att_gbs / peak_gbs if att_gbs else None, bytes_per_row=8 * W),
                                     layernorm=dict(achieved_gbs=ln_gbs, frac=ln_gbs / peak_gbs if ln_gbs else None, bytes_per_row="6W ln_1, 8W ln_2")))

    # ---- worst-case shape: every row truncated to 77 tokens (tokenizer.py:260-262), the shape SURVEY's target is defined on ----
    dense77 = None
    if not a.no_dense77:
        dset = eng.upload_captions(dense_caps) + (dense_anchor,)
        dd = draws(9000, dense_caps)
        device_step(*dd, cset=dset)
        torch.cuda.synchronize()
        rd = gemm_roofline(dd, dset, 2)
        d_tf = rd["gemm_flops"] / (rd["gemm_ms"] * 1e-3) / 1e12
        d_alg = float(sum(cfg.flops_for_length(int(x)) for x in rd["lens"]))
        dense77 = dict(value=cands_step / (rd["step_ms_timed"] * 1e-3), unit=UNIT, ms_per_step=rd["step_ms_timed"], steps=2,
                       gemm_tflops=d_tf, frac=d_tf / peak_tf, gemm_ms_per_step=rd["gemm_ms"], in_situ_ms_per_step=rd["insitu"],
                       rows_executed_per_step=int(rd["rows_exec"]), rows_without_prefix_sharing=int(rd["lens"].sum()),
                       mean_len=float(rd["lens"].mean()), whole_step_tflops=d_alg / (rd["step_ms_timed"] * 1e-3) / 1e12,
                       what="same device-resident step on 'dense-77' captions (40-60 words: every candidate row is 77 tokens), per GPU")
        del dset

    # ---- strong scaling with a collective ON the path (SURVEY.md 8e; BASELINE configs 3 and 4): ONE global batch of B captions
    #      over all ranks - sample-sharded (one all-gather of the winners per round) and candidate-sharded (one packed
    #      (loss, index) all-gather per phase + the winner rows), k = 1 and the k = 2 candidate-sharded shape ----
    global_batch = None
    if world > 1 and not a.no_global_batch:
        global_batch = {}
        gsteps = min(a.steps, 5)
        for mode, kk in (("samples", 1), ("candidates", 1), ("candidates", 2)):
            np.random.seed(4000)
            attack_text_leaf(tower, None, gcaps, ganchor.clone(), dev, objective="l2", n=n, k=kk, shard=mode)
            torch.cuda.synchronize()
            barrier()
            t0 = time.perf_counter()
            for i in range(gsteps):
                np.random.seed(4001 + i)
                gf, gadv = attack_text_leaf(tower, None, gcaps, ganchor.clone(), dev, objective="l2", n=n, k=kk, shard=mode)
                float(gf[0, 0].item())
            torch.cuda.synchronize()
            g_ms = torch.tensor([(time.perf_counter() - t0) * 1e3 / gsteps], dtype=torch.float64, device=dev)
            barrier()
            dist.all_reduce(g_ms, op=dist.ReduceOp.MAX)
            # every rank must hold the same global result
            h = torch.tensor([zlib.crc32("\x00".join(gadv).encode())], dtype=torch.int64, device=dev)
            hs = [torch.zeros_like(h) for _ in range(world)]
            dist.all_gather(hs, h)
            global_batch[f"{mode}_k{kk}"] = dict(value=2 * kk * B * n / (g_ms.item() * 1e-3), unit=UNIT, ms_per_step=g_ms.item(), scaling="strong",
                                                 global_batch=B, k=kk, steps=gsteps, ranks_agree=len({int(x.item()) for x in hs}) == 1)
        global_batch["what"] = ("attack_text_leaf(shard=...) end to end (host strings in, winners out) on ONE global batch over all ranks; "
                                "single-GPU e2e of the same call is the line's e2e.ms_per_step")

    # ---- per-rank record: which GPU is the straggler, and at what clock ----
    clk_sum = clk.summary()
    mine = torch.tensor([dev_ms_local / a.steps, e2e_ms_local / a.steps, float(clk_sum.get("sm_mhz") or 0)], dtype=torch.float64, device=dev)
    per_rank = [torch.zeros_like(mine) for _ in range(world)]
    if world > 1:
        dist.all_gather(per_rank, mine)
    else:
        per_rank = [mine]
    per_rank = dict(ms_per_step=[round(float(t[0]), 3) for t in per_rank], e2e_ms_per_step=[round(float(t[1]), 3) for t in per_rank],
                    sm_mhz=[int(t[2]) for t in per_rank])

    # the same executed FLOPs against the tensor peak AT THE CLOCK THE BOARD'S POWER CAP ALLOWED during the timed region
    # (SMs x 8192 dense bf16 FLOP per clock x the median SM clock nvidia-smi reported under load)
    if clk_sum.get("sm_mhz"):
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        cpeak = sms * 8192 * clk_sum["sm_mhz"] * 1e6 / 1e12
        roofline["clock_scaled_peak_tflops"] = cpeak
        roofline["frac_of_clock_scaled_peak"] = achieved / cpeak
        roofline["clock_scaled_note"] = ("achieved / (SMs x 8192 FLOP/clk x median SM clock under load): what the tensor pipe delivers of what the "
                                         "power-capped clock allows; ncu's sm__pipe_tensor_cycles_active reads 85-94 % on these GEMMs (profiles/r2_17_ncu_summary.txt)")
    h2d = int(sum(len(c) for c in caps) + 32 + 4 * (B + 1) + 3 * 4 * B * n) * k
    d2h = (2 * 4 * B + 4 + 4) * k
    line = dict(metric=METRIC, value=total_cands / (dev_ms * 1e-3), unit=UNIT, n_gpus=world, steps=a.steps, warmup=a.warmup,
                ms_per_step=step_ms, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16", data="synthetic",
                config=dict(workload=workload_name(a), candidates_per_step_per_gpu=cands_step, tower=a.model, width=W, layers=L,
                            rho=n, k=k, batch_per_gpu=B, captions=a.captions, l2="flushed between timed steps (256 MB write); "
                            "per-phase activations ~%.1f GB" % (rows_exec / 2 * W * 14 / 1e9), parallelism=f"dp{world} sample-sharded"),
                e2e=dict(value=total_cands / (e2e_ms * 1e-3), unit=UNIT, ms_per_step=e2e_ms / a.steps, h2d_bytes_per_step=h2d,
                         d2h_bytes_per_step=d2h),
                e2e_constrained=dict(value=total_cands / (con_ms * 1e-3), unit=UNIT, ms_per_step=con_ms / a.steps,
                                     what="attack_text_leaf(constrain=True): validity masks from leaf_constrain_mask (device), "
                                          "synthetic word list", sentences_changed_last_step=int(changed)),
                gpu_launches=int(launches), clocks=clk_sum, per_rank=per_rank, roofline=roofline)
    if train is not None:
        line["train_step"] = train
    if k4 is not None:
        line["k4"] = k4
    if dense77 is not None:
        line["dense77"] = dense77
    if global_batch is not None:
        line["global_batch"] = global_batch
    if rank == 0:
        if world == 1 and not a.no_library_baseline:
            try:
                line["gpu_library_baseline"] = gpu_library_baseline(a, tower.open_clip_state_dict(), caps, anchor, cfg, dev)
                lb = line["gpu_library_baseline"]
                lb["speedup_e2e_over_fp32_tf32"] = line["e2e"]["value"] / lb["fp32_tf32"]["e2e_candidates_per_s"]
                lb["speedup_e2e_over_bf16_autocast"] = line["e2e"]["value"] / lb["bf16_autocast"]["e2e_candidates_per_s"]
                lb["speedup_device_over_bf16_autocast"] = line["value"] / lb["bf16_autocast"]["device_candidates_per_s"]
            except Exception as ex:
                line["gpu_library_baseline"] = dict(failed=repr(ex))
        if world == 1 and not a.no_cpu_baseline:
            try:
                line["cpu_baseline"], _, _ = cpu_attack_rate(a, seconds=a.cpu_seconds)
            except Exception as ex:                          # the baseline must never take the bench line down
                line["cpu_baseline"] = dict(value=None, unit=UNIT, cores=os.cpu_count(), kind="port", sample=f"failed: {ex}")
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)

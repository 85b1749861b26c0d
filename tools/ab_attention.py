"""Timing of the attention kernel alone on the bench workload's real sequence shapes.

    python tools/ab_attention.py

Builds the packed-row metadata of both attack phases of the ViT-H bench workload on the host (same rule as
prefix_kernel / meta_kernel, without duplicate elimination), fills qkv with random bf16 and times leaf_test_attention
with CUDA events. To compare two builds, run it once per build with LEAF_B200_LIB naming the library.
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from leaf_b200 import synth                                  # noqa: E402
from leaf_b200.attack import V_DEFAULT                       # noqa: E402
from leaf_b200.tower import LeafTextTower                    # noqa: E402


def host_meta(tok, ln, base):
    tok, ln, base = tok.cpu().numpy(), ln.cpu().numpy(), base.cpu().numpy()
    N = len(ln)
    t = np.clip(ln, 1, 77)
    p = np.zeros(N, dtype=np.int64)
    for i in range(N):
        b = base[i]
        if b >= 0 and b != i:
            lim = min(t[i], t[b])
            d = np.nonzero(tok[i, :lim] != tok[b, :lim])[0]
            p[i] = min(d[0] if len(d) else lim, t[i] - 1)
    own = t - p
    cu = np.concatenate([[0], np.cumsum(own)])
    brow = np.where((p > 0) & (base >= 0), cu[np.maximum(base, 0)], cu[:-1])
    meta = np.stack([cu[:-1], t, p, brow], axis=1).astype(np.int32)
    return meta, int(cu[-1])


def main():
    dev = torch.device("cuda", 0)
    B, n = 128, 50
    caps = synth.make_captions(B, seed=100, kind="typical")
    H, W = 16, 1024
    cfg = synth.TowerCfg("ab", W, 1, H, 1024)               # the kernel only depends on heads and width
    eng = LeafTextTower.random(cfg, seed=0, device=dev).leaf_engine
    assert eng.width == W and eng.heads == H, (eng.width, eng.heads)
    rs = np.random.RandomState(0)
    Vt = np.asarray(V_DEFAULT, dtype=np.int32)
    pos = np.stack([rs.choice(range(2 * len(S) + 1), size=n, replace=n > 2 * len(S) + 1) for S in caps]).astype(np.int32)
    ch = Vt[np.stack([rs.choice(range(len(Vt)), size=n, replace=False) for _ in caps])]
    d, o = eng.upload_captions(caps)
    space = torch.full((B * n,), 32, dtype=torch.int32, device=dev)
    phases = []
    tok, ln, base = eng.expand_tokenize(d, o, B, n, pos=torch.from_numpy(pos).to(dev), chr_=space)
    phases.append(host_meta(tok, ln, base))
    sel = torch.from_numpy(rs.randint(0, n, size=B).astype(np.int32)).to(dev)
    tok, ln, base = eng.expand_tokenize(d, o, B, n, pos=torch.from_numpy(pos).to(dev), chr_=torch.from_numpy(ch).to(dev), sel=sel)
    phases.append(host_meta(tok, ln, base))
    for ph, (meta, rows) in enumerate(phases):
        meta_d = torch.from_numpy(meta).to(dev)
        qkv = (torch.randn((rows, 3 * W), device=dev) * 0.5).to(torch.bfloat16)
        out = eng.test_attention(qkv, meta_d)
        times = []
        for rep in range(6):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(10):
                eng.test_attention(qkv, meta_d, out)
            b.record()
            torch.cuda.synchronize()
            if rep:
                times.append(a.elapsed_time(b) / 10)
        nkt = ((np.minimum(meta[:, 1] - 1, 76)) >> 4) + 1
        print(f"phase {ph + 1}: rows={rows} seqs={len(meta)} mean t={meta[:, 1].mean():.1f} mean own={(meta[:, 1] - meta[:, 2]).mean():.1f} "
              f"nkt hist={np.bincount(nkt, minlength=6)[1:].tolist()}")
        ms = np.array(times)
        gb = rows * W * 8 / 1e9
        print(f"  {ms.mean() * 1e3:8.1f} us  (min {ms.min() * 1e3:.1f})  {gb / ms.mean() * 1e3 / 1e3:.2f} TB/s algorithmic")


if __name__ == "__main__":
    main()

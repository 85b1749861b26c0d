"""Kernels launched per engine call (leaf_launch_count, which bench.py reports as gpu_launches), on a small random tower with
L layers in the open_clip layout (fused in_proj) and in the HF layout (split q / k / v)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _engine(layout):
    from leaf_b200.engine import LeafEngine
    from leaf_b200.tower import LeafTextTower, open_clip_to_hf
    tower = LeafTextTower.random("small", seed=5)
    if layout == "open_clip":
        return tower.leaf_engine, tower.open_clip_state_dict()
    sd = open_clip_to_hf(tower.open_clip_state_dict())
    return LeafEngine(sd, heads=tower.heads), sd


@pytest.mark.parametrize("layout", ["open_clip", "hf"])
def test_launch_counts(layout):
    from leaf_b200 import synth
    eng, sd = _engine(layout)
    L, hf = eng.layers, layout == "hf"

    def count(f):
        eng.launch_count(reset=True)
        f()
        return eng.launch_count()

    caps = synth.make_captions(6, seed=2)
    B, n = len(caps), 8
    rs = np.random.RandomState(0)
    pos = torch.from_numpy(np.stack([rs.randint(0, 2 * len(S) + 1, size=n) for S in caps]).astype(np.int32)).cuda()
    V = np.asarray(synth.V_DEFAULT, dtype=np.int32)
    chr_ = torch.from_numpy(V[rs.randint(0, len(V), size=(B, n))]).cuda()
    d, o = eng.upload_captions(caps)
    assert count(lambda: eng.expand_tokenize(d, o, B, 0)) == 1
    tok, ln, base = eng.expand_tokenize(d, o, B, n, pos, chr_)
    eng.check_status()

    assert count(lambda: eng.encode_tokens(tok, ln)) == 7 * L + 9
    assert count(lambda: eng.encode_tokens(tok, ln, normalize=True)) == 7 * L + 10
    assert count(lambda: eng.encode_tokens(tok, ln, base=base, dedup=(B * n, n))) == 7 * L + 10
    assert count(lambda: eng.encode_tokens(tok, ln, base=base, dedup=(B * n, n), trim=True)) == 7 * L + 11
    eng.set_prune_last(False)
    try:
        assert count(lambda: eng.encode_tokens(tok, ln)) == 7 * L + 8
    finally:
        eng.set_prune_last(True)

    rows, lengths = eng.tokenize(caps, with_lengths=True)
    assert count(lambda: eng.forward_train(rows)) == 7 * L + 6
    grads = {k: torch.zeros_like(v) for k, v in sd.items()}
    dfeat = torch.randn((B, eng.embed_dim), device="cuda")
    assert count(lambda: eng.backward(dfeat, grads)) == (15 if hf else 13) * L + 6
    assert count(lambda: eng.forward_train(rows, host_lengths=lengths)) == 7 * L + 7
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        assert count(lambda: eng.backward(dfeat, grads)) == (15 if hf else 13) * L + 7
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=warn)

    assert count(eng.refresh_weights) == (6 if hf else 4) * L + 2

    eng.load_words(["a", "photo", "of", "the", "dog", "cat"])
    assert count(lambda: eng.constrain_mask(d, o, B, n, pos, chr_)) == 2
    feats = eng.encode_tokens(tok, ln)
    anchor = torch.randn((B, eng.embed_dim), device="cuda")
    assert count(lambda: eng.score(feats[:B * n], anchor, B, n)) == 1
    assert count(lambda: eng.topk(feats[:, 0].contiguous(), 5)) == 1
    torch.cuda.synchronize()

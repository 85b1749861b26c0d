"""Deterministic mode of the K4 backward (leaf_set_deterministic, switched by torch.use_deterministic_algorithms): every
gradient the engine writes, and the gradient-norm reduction, must be a function of the inputs alone, bit for bit - across
repeated runs, SM budgets, dependent launch on or off, and engines built from the same weights. Every check runs with
torch's flag on and restores it afterwards. "Bit-equal" compares int32 views, so -0.0 and NaN payloads count."""
import contextlib

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

WIDE = None          # a ViT-H-wide tower (W = 1024, 16 heads, E = 1024) with two layers, built on first use


def _tower_cfg(name):
    from leaf_b200 import synth
    global WIDE
    if name != "wide":
        return synth.TOWERS[name]
    if WIDE is None:
        WIDE = synth.TowerCfg("ViT-H-width", 1024, 2, 16, 1024)
    return WIDE


@contextlib.contextmanager
def _torch_deterministic(on=True):
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(on)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=warn)


@pytest.fixture(autouse=True)
def deterministic():
    with _torch_deterministic():
        yield


def _bits(t):
    return t.contiguous().view(torch.int32)


def _bit_equal(a, b):
    return torch.equal(_bits(a), _bits(b))


def _batches():
    from leaf_b200 import synth
    one = synth.make_captions(1, seed=31)[0]
    return {"repeated": [one] * 128,                                          # 128 rows share every token id
            "mixed": synth.make_captions(5, seed=32) + synth.make_captions(1, seed=33, kind="dense-77") + ["", "a"],
            "single": [one]}


def _grads_of(tower, tok, w):
    tower.zero_grad()
    f = tower.encode_text(tok)
    (f * w).sum().backward()
    return tower.flat_grads.clone()


@pytest.mark.parametrize("name,quick", [("small", False), ("tiny", True), ("wide", False)])
def test_repeated_backward_is_bit_equal(name, quick):
    from leaf_b200 import synth
    from leaf_b200.tower import LeafTextTower
    cfg = _tower_cfg(name)
    tower = LeafTextTower(synth.random_tower_state_dict(cfg, seed=21, device="cuda"), heads=cfg.heads, quick_gelu=quick).trainable()
    for kind, caps in _batches().items():
        tok = tower.tokenizer(caps)
        w = torch.randn((len(caps), cfg.embed_dim), generator=torch.Generator(device="cuda").manual_seed(5), device="cuda")
        first = _grads_of(tower, tok, w)
        assert float(first.abs().max()) > 0
        for i in range(4):
            assert _bit_equal(first, _grads_of(tower, tok, w)), (name, kind, i)


@pytest.mark.parametrize("name", ["small", "wide"])
def test_sm_budget_and_dependent_launch_change_no_bit(name, monkeypatch):
    from leaf_b200 import synth
    from leaf_b200.tower import LeafTextTower
    cfg = _tower_cfg(name)
    sd = synth.random_tower_state_dict(cfg, seed=6, device="cuda")
    monkeypatch.setenv("LEAF_PDL", "0")
    plain = LeafTextTower({k: v.clone() for k, v in sd.items()}, heads=cfg.heads).trainable()
    monkeypatch.delenv("LEAF_PDL")
    chained = LeafTextTower({k: v.clone() for k, v in sd.items()}, heads=cfg.heads).trainable()
    caps = synth.make_captions(24, seed=8) + synth.make_captions(2, seed=9, kind="dense-77")
    tok = chained.tokenizer(caps)
    w = torch.randn((len(caps), cfg.embed_dim), generator=torch.Generator(device="cuda").manual_seed(7), device="cuda")
    want = _grads_of(plain, tok, w)
    eng = chained.leaf_engine
    for budget in (0, 64, 32, 0):
        with eng.sm_budget(budget):
            assert _bit_equal(want, _grads_of(chained, tok, w)), budget


def _frozen(grads):
    """Half of the parameters frozen (None): the LayerNorms, both embeddings, every MLP input weight."""
    out = dict(grads)
    for k in out:
        if any(s in k for s in ("ln_", "layer_norm", "embedding", "c_fc.weight", "fc1.weight")):
            out[k] = None
    return out


@pytest.mark.parametrize("layout", ["open_clip", "hf"])
@pytest.mark.parametrize("frozen", [False, True])
def test_two_engines_from_one_state_dict_agree_to_the_bit(layout, frozen):
    from leaf_b200 import synth
    from leaf_b200.engine import LeafEngine
    from leaf_b200.tower import open_clip_to_hf
    cfg = synth.TOWERS["small"]
    sd = synth.random_tower_state_dict(cfg, seed=4, device="cuda")
    if layout == "hf":                   # q / k / v split, [E, W] projection (split-K projection weight gradient)
        sd = open_clip_to_hf(sd)
    tok = LeafEngine(sd, heads=cfg.heads).tokenize(synth.make_captions(12, seed=1) + ["", "a"])
    d = torch.randn((tok.shape[0], cfg.embed_dim), generator=torch.Generator(device="cuda").manual_seed(3), device="cuda")
    res = []
    for _ in range(2):
        eng = LeafEngine({k: v.clone() for k, v in sd.items()}, heads=cfg.heads)
        g = {k: torch.zeros_like(v) for k, v in sd.items()}
        if frozen:
            g = _frozen(g)
        f = eng.forward_train(tok)
        eng.backward(d, g, eng.last_generation)
        assert eng.deterministic
        res.append((f, g))
    assert _bit_equal(res[0][0], res[1][0])
    assert (None in res[0][1].values()) == frozen
    for k, g0 in res[0][1].items():
        if g0 is not None:
            assert float(g0.abs().max()) > 0, k
            assert _bit_equal(g0, res[1][1][k]), k


@pytest.mark.parametrize("name,quick", [("small", False), ("tiny", True)])
def test_deterministic_gradients_meet_the_autograd_bars(name, quick):
    from leaf_b200 import synth
    from leaf_b200.tower import LeafTextTower
    from tests.test_gpu_backward import _ref_grads
    cfg = synth.TOWERS[name]
    sd = synth.random_tower_state_dict(cfg, seed=11, exact_numpy=True)
    tower = LeafTextTower(sd, heads=cfg.heads, quick_gelu=quick).trainable()
    caps = synth.make_captions(6, seed=5) + synth.make_captions(1, seed=5, kind="dense-77") + ["a", ""]
    tok = tower.tokenizer(caps)
    g = torch.Generator().manual_seed(0)
    with torch.no_grad():
        anchor = tower.encode_text(tok) + 0.3 * torch.randn((len(caps), cfg.embed_dim), generator=g).cuda()
    tower.zero_grad()
    f = tower.encode_text(tok)
    torch.nn.functional.mse_loss(anchor, f, reduction="none").sum(-1).mean().backward()
    assert tower.leaf_engine.deterministic
    det = tower.flat_grads.clone()
    with _torch_deterministic(False):                  # the fp32 autograd reference, and the engine's default mode
        cot = (2.0 * (f.detach() - anchor) / len(caps)).contiguous()
        _, _, vjp = _ref_grads(sd, tok, anchor, cfg.heads, quick, cotangent=cot)
        tower.zero_grad()
        f2 = tower.encode_text(tok)
        torch.nn.functional.mse_loss(anchor, f2, reduction="none").sum(-1).mean().backward()
        assert not tower.leaf_engine.deterministic
        default = tower.flat_grads.clone()
    assert torch.equal(f.detach(), f2.detach())
    for k, safe in tower._names.items():
        off, n, shape = tower._slices[k]
        got, want = det[off:off + n].view(shape), vjp[k]
        rel = ((got - want).norm() / want.norm().clamp_min(1e-20)).item()
        cos = torch.nn.functional.cosine_similarity(got.flatten().double(), want.flatten().double(), dim=0).item()
        assert rel <= 3e-2 and cos >= 0.999, (k, rel, cos)
    assert ((det - default).norm() / default.norm()).item() <= 1e-5


def test_sumsq_is_reproducible_and_accurate():
    from leaf_b200.tower import LeafTextTower
    eng = LeafTextTower.random("tiny", seed=0).leaf_engine
    eng.set_deterministic(True)
    g = torch.randn(3_000_004, generator=torch.Generator(device="cuda").manual_seed(2), device="cuda")
    g[::7] *= 1e-3
    outs = []
    for _ in range(4):
        out = torch.zeros(1, device="cuda")
        eng.sumsq(g, out)
        outs.append(out)
    assert all(_bit_equal(outs[0], o) for o in outs[1:])
    want = (g.double() ** 2).sum().item()
    assert abs(outs[0].item() - want) <= 1e-6 * want, (outs[0].item(), want)


@pytest.mark.parametrize("budget", [None, 64])
def test_fare_trainer_steps_are_bit_reproducible(budget):
    """Two FareTrainers from one state dict, accumulation over two micro-batches and clipping: parameters, both AdamW moments
    and the adversarial texts are bit-equal after every optimizer step. budget: the second trainer's engine runs with its GEMM
    grids capped at 64 SMs (leaf_set_sm_budget) throughout."""
    from leaf_b200 import synth
    from leaf_b200.fare import FareTrainer
    from leaf_b200.tower import LeafTextTower
    cfg = synth.TOWERS["small"]
    sd = synth.random_tower_state_dict(cfg, seed=3, exact_numpy=True)
    frozen = LeafTextTower(synth.perturbed_copy(sd, seed=4, std=1e-2, exact_numpy=True), heads=cfg.heads)
    hp = dict(rho=12, k_adv=1, accum_freq=2, grad_clip_norm=0.5, lr=1e-3, wd=0.05)
    trs = [FareTrainer(LeafTextTower(sd, heads=cfg.heads), frozen, **hp),
           FareTrainer(LeafTextTower(sd, heads=cfg.heads), frozen, backward_sm_budget=budget, **hp)]
    with trs[1].tower.leaf_engine.sm_budget(budget or 0):
        for i in range(6):
            texts = synth.make_captions(6, seed=40 + i)
            adv = []
            for tr in trs:
                np.random.seed(100 + i)
                adv.append(tr.step(texts)[1])
            assert adv[0] == adv[1], i
            if i % 2 == 1:
                a, b = trs
                assert a.opt_step == b.opt_step == (i + 1) // 2
                assert _bit_equal(a.tower.flat_params, b.tower.flat_params), i
                assert _bit_equal(a.exp_avg, b.exp_avg), i
                assert _bit_equal(a.exp_avg_sq, b.exp_avg_sq), i
    assert not torch.equal(trs[0].tower.flat_params, LeafTextTower(sd, heads=cfg.heads).flat_params)


def test_fare_trainer_with_charmer_runs_under_deterministic_mode():
    """use_charmer=True (the single-sentence Charmer attack inside the step) raises no torch determinism error and is
    reproducible as well."""
    from leaf_b200 import synth
    from leaf_b200.fare import FareTrainer
    from leaf_b200.tower import LeafTextTower
    cfg = synth.TOWERS["tiny"]
    sd = synth.random_tower_state_dict(cfg, seed=8, exact_numpy=True)
    frozen = LeafTextTower(synth.perturbed_copy(sd, seed=9, std=1e-2, exact_numpy=True), heads=cfg.heads, quick_gelu=True)
    trs = [FareTrainer(LeafTextTower(sd, heads=cfg.heads, quick_gelu=True), frozen, rho=8, k_adv=1, use_charmer=True,
                       grad_clip_norm=1.0, lr=1e-3) for _ in range(2)]
    texts = synth.make_captions(3, seed=50)
    adv = []
    for tr in trs:
        np.random.seed(7)
        adv.append(tr.step(texts)[1])
    assert adv[0] == adv[1]
    assert _bit_equal(trs[0].tower.flat_params, trs[1].tower.flat_params)

"""Checkpoint and resume of FARE training: FareTrainer.state_dict / load_state_dict (an interrupted and resumed run equals an
uninterrupted one bit for bit under torch.use_deterministic_algorithms), LeafTextTower.load_state_dict /
load_open_clip_state_dict (the engine computes with the loaded weights), and the reference's epoch checkpoint
{epoch, name, state_dict, optimizer} in both directions (train_AT_text_only.py:351-372, 516-525, 560-569). "Bit-equal" compares
int32 views, so -0.0 and NaN payloads count."""
import contextlib
from collections import OrderedDict

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

HP = dict(rho=12, k_adv=1, accum_freq=2, grad_clip_norm=0.5, lr=1e-3, wd=0.05)
SEED = 123
TOWERS = [("small", False), ("tiny", True)]


@contextlib.contextmanager
def _torch_deterministic(on):
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(on)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=warn)


def _bit_equal(a, b):
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def _batches():
    from leaf_b200 import synth
    return [synth.make_captions(6, seed=40 + i) for i in range(6)]


def _pretrained(name, seed=3):
    from leaf_b200 import synth
    cfg = synth.TOWERS[name]
    return cfg, synth.random_tower_state_dict(cfg, seed=seed, exact_numpy=True)


def _trainer(name, quick, seed=3, **hp):
    """A FareTrainer on the `name` tower initialised from `seed`; the frozen anchor tower is always the same pretrained model."""
    from leaf_b200 import synth
    from leaf_b200.fare import FareTrainer
    from leaf_b200.tower import LeafTextTower
    cfg, base = _pretrained(name)
    frozen = LeafTextTower(synth.perturbed_copy(base, seed=4, std=1e-2, exact_numpy=True), heads=cfg.heads, quick_gelu=quick)
    _, sd = _pretrained(name, seed)
    return FareTrainer(LeafTextTower(sd, heads=cfg.heads, quick_gelu=quick), frozen, **{**HP, **hp})


def _state_tensors(tr):
    return {"params": tr.tower.flat_params, "exp_avg": tr.exp_avg, "exp_avg_sq": tr.exp_avg_sq, "grads": tr.tower.flat_grads}


@pytest.mark.parametrize("name,quick", TOWERS)
def test_interrupted_run_resumes_bit_for_bit(name, quick, tmp_path):
    """Accumulation over two micro-batches with clipping, six micro-batches, one numpy seed for the whole run: run A is
    uninterrupted; run B stops after micro-batch 3 (inside a window) or 4 (at a window boundary), saves, and continues in a
    trainer whose tower was initialised from another seed, after the numpy stream was moved elsewhere."""
    batches = _batches()
    with _torch_deterministic(True):
        np.random.seed(SEED)
        a = _trainer(name, quick)
        out_a = [a.step(t) for t in batches]
        for stop in (3, 4):
            np.random.seed(SEED)
            b = _trainer(name, quick)
            for t in batches[:stop]:
                b.step(t)
            state = b.state_dict()
            assert (state["grads"] is None) == (stop % 2 == 0)
            torch.save(state, tmp_path / "state.pt")
            del b, state
            np.random.seed(999)
            b = _trainer(name, quick, seed=77)
            assert not torch.equal(b.tower.flat_params, a.tower.flat_params)
            b.load_state_dict(torch.load(tmp_path / "state.pt"))
            assert (b.opt_step, b.micro) == (stop // 2, stop)
            for i, t in enumerate(batches[stop:], start=stop):
                loss, adv = b.step(t)
                assert adv == out_a[i][1], (stop, i)
                assert _bit_equal(loss, out_a[i][0]), (stop, i, loss.item(), out_a[i][0].item())
            assert a.opt_step == b.opt_step == 3
            for what, ta in _state_tensors(a).items():
                assert _bit_equal(ta, _state_tensors(b)[what]), (stop, what)
    assert not torch.equal(a.tower.flat_params, _trainer(name, quick).tower.flat_params)        # training moved the weights


def test_resume_without_deterministic_mode(tmp_path):
    """Default (atomic) gradient sums: the resumed trainer starts from bit-equal state, so its first step draws the same
    adversarial texts as the interrupted run continuing on its own; the update then agrees to the tolerance of
    test_fare_trainer_matches_a_torch_loop."""
    batches = _batches()
    _, sd = _pretrained("small")
    with _torch_deterministic(False):
        np.random.seed(SEED)
        b = _trainer("small", False)
        for t in batches[:3]:
            b.step(t)
        torch.save(b.state_dict(), tmp_path / "state.pt")
        loss_b, adv_b = b.step(batches[3])                      # the uninterrupted continuation: completes the window
        np.random.seed(999)
        c = _trainer("small", False, seed=77)
        c.load_state_dict(torch.load(tmp_path / "state.pt"))
        loss_c, adv_c = c.step(batches[3])
    assert adv_b == adv_c
    assert torch.allclose(loss_b, loss_c, rtol=1e-5)
    assert b.opt_step == c.opt_step == 2
    for (k, pb), (_, pc) in zip(b.tower.named_tower_parameters(), c.tower.named_tower_parameters()):
        upd = (pb - sd[k].cuda()).norm().clamp_min(1e-12)
        assert ((pb - pc).norm() / upd).item() < 2e-2, k
        assert ((pb - pc).abs() > 1e-6 + 1e-4 * pb.abs()).float().mean().item() < 1e-3, k
    for mb, mc in ((b.exp_avg, c.exp_avg), (b.exp_avg_sq, c.exp_avg_sq)):
        assert ((mb - mc).norm() / mb.norm()).item() < 1e-3


def test_state_without_rng_restores_everything_else(tmp_path):
    """include_rng=False: every tensor and counter comes back bit-equal, the numpy stream is left where it is, and with the
    stream set alike the two trainers go on to draw the same candidates."""
    batches = _batches()
    with _torch_deterministic(True):
        np.random.seed(SEED)
        b = _trainer("small", False)
        for t in batches[:3]:
            b.step(t)
        state = b.state_dict(include_rng=False)
        assert state["numpy_rng"] is None
        torch.save(state, tmp_path / "state.pt")
        np.random.seed(999)
        before = np.random.get_state()
        c = _trainer("small", False, seed=77)
        c.load_state_dict(torch.load(tmp_path / "state.pt"))
        after = np.random.get_state()
        assert np.array_equal(before[1], after[1]) and before[2] == after[2]
        assert (c.opt_step, c.micro) == (b.opt_step, b.micro) == (1, 3)
        for what, tb in _state_tensors(b).items():
            assert _bit_equal(tb, _state_tensors(c)[what]), what
        out = []
        for tr in (b, c):
            np.random.seed(5)
            out.append(tr.step(batches[3]))
    assert out[0][1] == out[1][1] and _bit_equal(out[0][0], out[1][0])


@pytest.mark.parametrize("name,quick", TOWERS)
def test_tower_loads_refresh_the_engine(name, quick):
    """After LeafTextTower.load_state_dict or load_open_clip_state_dict, the inference and the training forward equal those of
    a tower constructed from the loaded weights, bit for bit; the flat buffer and the .grad views stay where they were."""
    from leaf_b200 import synth
    from leaf_b200.tower import LeafTextTower
    cfg, sd_a = _pretrained(name, 1)
    sds = {s: _pretrained(name, s)[1] for s in (2, 3)}
    t = LeafTextTower(sd_a, heads=cfg.heads, quick_gelu=quick).trainable()
    t.attach_grads()
    ptrs = [t.flat_params.data_ptr()] + [p.grad.data_ptr() for _, p in t.named_tower_parameters()]
    tok = t.tokenizer(synth.make_captions(10, seed=6) + synth.make_captions(2, seed=6, kind="dense-77"))

    def features(tower):
        with torch.no_grad():
            return tower.encode_text(tok), tower.leaf_engine.forward_train(tok)

    f_a = features(t)
    for s, load in ((2, lambda sd, ref: t.load_state_dict(ref.state_dict())),
                    (3, lambda sd, ref: t.load_open_clip_state_dict({**{"text." + k: v for k, v in sd.items()},
                                                                     "visual.proj": torch.zeros(4), "logit_scale": torch.ones([])})),
                    (1, lambda sd, ref: t.load_open_clip_state_dict({"module." + k: v.cuda() for k, v in sd.items()}))):
        sd = sd_a if s == 1 else sds[s]
        ref = LeafTextTower(sd, heads=cfg.heads, quick_gelu=quick)
        want = features(ref)
        load(sd, ref)
        got = features(t)
        assert all(_bit_equal(g, w) for g, w in zip(got, want)), s
        assert s == 1 or not _bit_equal(got[0], f_a[0])
    assert ptrs == [t.flat_params.data_ptr()] + [p.grad.data_ptr() for _, p in t.named_tower_parameters()]

    before = t.flat_params.clone()
    key = "transformer.resblocks.1.mlp.c_fc.bias"
    cases = [({k: v for k, v in sds[2].items() if k != key}, f"missing: {key}"),
             ({**sds[2], "ln_final.weight": sds[2]["ln_final.weight"][:-1]}, "shape of ln_final.weight"),
             ({**sds[2], "transformer.resblocks.9.ln_1.weight": sds[2]["ln_final.weight"]}, "unexpected: transformer.resblocks.9.ln_1.weight")]
    for bad, msg in cases:
        with pytest.raises(ValueError, match=msg.replace(".", r"\.")):
            t.load_open_clip_state_dict(bad)
    assert torch.equal(t.flat_params, before)                   # a refused state dict changes nothing
    with pytest.raises(RuntimeError, match=key.replace(".", "__")):
        t.load_state_dict({k: v for k, v in t.state_dict().items() if k != key.replace(".", "__")})
    with pytest.raises(ValueError, match="assign"):
        t.load_state_dict(t.state_dict(), assign=True)


# ---- the reference's epoch checkpoint -------------------------------------------------------------------------------------
def _clip(seed, quick=False):
    """An open_clip-named CLIP: the text tower at the top level (tests/test_gpu_dropin.py's module), logit_scale, and a
    small visual stub under `visual.`."""
    from leaf_b200 import synth
    from tests.test_gpu_dropin import OpenClipNamedTower

    class Clip(OpenClipNamedTower):
        def __init__(self):
            super().__init__(synth.TOWERS["small"], quick=quick, seed=seed)
            self.visual = torch.nn.Sequential(OrderedDict([("conv1", torch.nn.Conv2d(3, 8, 4, bias=False)), ("ln_pre", torch.nn.LayerNorm(8)),
                                                           ("proj", torch.nn.Linear(8, 256))]))
            g = torch.Generator().manual_seed(seed)
            with torch.no_grad():
                for p in self.visual.parameters():
                    p.copy_(torch.randn(p.shape, generator=g))
                self.logit_scale.fill_(float(np.log(1 / 0.07)) + seed)

    return Clip().cuda()


def _holder(model, holder):
    from tests.test_gpu_dropin import _DDPLike
    return _DDPLike(model) if holder == "ddp" else model


def _reference_groups(model):
    """train_AT_text_only.py:326-341: (name, parameter) lists of the weight-decay-0 group and the rest."""
    exclude = lambda n, p: p.ndim < 2 or "bn" in n or "ln" in n or "bias" in n or "logit_scale" in n
    named = list(model.named_parameters())
    return [(n, p) for n, p in named if exclude(n, p)], [(n, p) for n, p in named if not exclude(n, p)]


def _reference_adamw(model, lr, wd, beta1, beta2, eps):
    g0, g1 = _reference_groups(model)
    return torch.optim.AdamW([{"params": [p for _, p in g0], "weight_decay": 0.0}, {"params": [p for _, p in g1], "weight_decay": wd}],
                             lr=lr, betas=(beta1, beta2), eps=eps)


def _text_params(model, tower):
    return {k: p for k, p in model.named_parameters() if k in tower._slices}


@pytest.mark.parametrize("holder", ["clip", "ddp"])
def test_reference_checkpoint_export(holder, tmp_path):
    from leaf_b200 import synth
    from leaf_b200.fare import FareTrainer
    from leaf_b200.tower import LeafTextTower, text_tower_state_dict
    cfg = synth.TOWERS["small"]
    model = _clip(31)
    sd = text_tower_state_dict(model.state_dict())
    frozen = LeafTextTower(synth.perturbed_copy(sd, seed=4, std=1e-2), heads=cfg.heads)
    hp = dict(lr=1e-3, wd=0.05, beta1=0.9, beta2=0.98, eps=1e-6)
    tr = FareTrainer(LeafTextTower(sd, heads=cfg.heads), frozen, rho=12, k_adv=1, **hp)
    np.random.seed(0)
    for t in _batches()[:2]:
        tr.step(t)
    wrapped = _holder(model, holder)
    torch.save(tr.reference_checkpoint(wrapped, epoch=2, name="leaf"), tmp_path / "epoch_latest.pt")
    ckpt = torch.load(tmp_path / "epoch_latest.pt")
    assert set(ckpt) == {"epoch", "name", "state_dict", "optimizer"} and (ckpt["epoch"], ckpt["name"]) == (2, "leaf")
    assert list(ckpt["state_dict"]) == list(wrapped.state_dict())

    fresh = _clip(32)
    fresh_w = _holder(fresh, holder)
    fresh_w.load_state_dict(ckpt["state_dict"], strict=True)
    opt = _reference_adamw(fresh_w, **hp)
    opt.load_state_dict(ckpt["optimizer"])
    trained, m, v = (tr._by_name(x) for x in (tr.tower.flat_params, tr.exp_avg, tr.exp_avg_sq))
    text = _text_params(fresh, tr.tower)
    assert len(text) == len(trained) == len(opt.state)           # the visual parameters and logit_scale have no state
    for k, p in text.items():
        assert _bit_equal(p.detach(), trained[k]), k
        st = opt.state[p]
        assert int(st["step"]) == tr.opt_step == 2
        assert _bit_equal(st["exp_avg"], m[k]) and _bit_equal(st["exp_avg_sq"], v[k]), k
    for k, p in model.named_parameters():
        if k not in text:
            assert torch.equal(dict(fresh.named_parameters())[k], p), k

    # one more step from the exported state: torch.optim.AdamW against leaf_adamw on the same gradients
    g = torch.Generator(device="cuda").manual_seed(9)
    grads = tr._by_name(tr.tower.flat_grads)
    for k, p in text.items():
        p.grad = torch.randn(p.shape, generator=g, device="cuda") * 1e-2
        grads[k].copy_(p.grad)
    opt.step()
    tr.optimizer_step()
    for k, p in text.items():
        assert torch.allclose(trained[k], p.detach(), rtol=1e-5, atol=1e-7), (k, (trained[k] - p).abs().max().item())
        assert torch.allclose(m[k], opt.state[p]["exp_avg"], rtol=1e-5, atol=1e-9), k


@pytest.mark.parametrize("holder", ["clip", "ddp"])
def test_reference_checkpoint_import(holder, tmp_path):
    from leaf_b200 import synth
    from leaf_b200.fare import FareTrainer
    from leaf_b200.tower import LeafTextTower, text_tower_state_dict
    cfg = synth.TOWERS["small"]
    hp = dict(lr=1e-3, wd=0.05, beta1=0.9, beta2=0.98, eps=1e-6)
    model = _clip(31)
    wrapped = _holder(model, holder)
    opt = _reference_adamw(wrapped, **hp)
    g = torch.Generator(device="cuda").manual_seed(2)
    for _ in range(3):
        for p in wrapped.parameters():
            p.grad = torch.randn(p.shape, generator=g, device="cuda") * 1e-2
        opt.step()
    torch.save({"epoch": 3, "name": "leaf", "state_dict": wrapped.state_dict(), "optimizer": opt.state_dict(),
                "scaler": {"scale": 65536.0}}, tmp_path / "epoch_3.pt")
    ckpt = torch.load(tmp_path / "epoch_3.pt")
    if holder == "ddp":
        assert all(k.startswith("module.") for k in ckpt["state_dict"])

    frozen = LeafTextTower(synth.random_tower_state_dict(cfg, seed=8, device="cuda"), heads=cfg.heads)
    tr = FareTrainer(LeafTextTower(synth.random_tower_state_dict(cfg, seed=5, device="cuda"), heads=cfg.heads), frozen, rho=12,
                     k_adv=1, accum_freq=2, **hp)
    tr.load_reference_checkpoint(ckpt, wrapped)
    assert (tr.opt_step, tr.micro) == (3, 6)
    trained, m, v = (tr._by_name(x) for x in (tr.tower.flat_params, tr.exp_avg, tr.exp_avg_sq))
    text = _text_params(model, tr.tower)
    assert len(text) == len(trained)
    for k, p in text.items():
        assert _bit_equal(trained[k], p.detach()), k
        assert _bit_equal(m[k], opt.state[p]["exp_avg"]) and _bit_equal(v[k], opt.state[p]["exp_avg_sq"]), k
    tok = tr.tower.tokenizer(synth.make_captions(8, seed=3))
    with torch.no_grad():
        want = LeafTextTower(text_tower_state_dict(model.state_dict()), heads=cfg.heads).encode_text(tok)
        assert _bit_equal(tr.tower.encode_text(tok), want)

    other = FareTrainer(LeafTextTower(synth.random_tower_state_dict(cfg, seed=6, device="cuda"), heads=cfg.heads), frozen, **hp)
    before = other.tower.flat_params.clone()
    for attr, val, key in (("lr", 2e-3, "lr"), ("wd", 0.1, "weight_decay"), ("beta2", 0.999, "betas"), ("eps", 1e-8, "eps")):
        old = getattr(other, attr)
        setattr(other, attr, val)
        with pytest.raises(ValueError, match=f"group [01] {key}"):
            other.load_reference_checkpoint(ckpt, wrapped)
        setattr(other, attr, old)
    names = [n for group in _reference_groups(wrapped) for n, _ in group]            # the optimizer's parameter ids, in order
    pid = next(i for i, n in enumerate(names) if n.endswith("transformer.resblocks.0.ln_1.weight"))
    ckpt["optimizer"]["state"][pid]["step"] = torch.tensor(2.0)
    with pytest.raises(ValueError, match="steps disagree"):
        other.load_reference_checkpoint(ckpt, wrapped)
    assert other.opt_step == 0 and torch.equal(other.tower.flat_params, before)


def test_state_of_another_tower_is_refused():
    small = _trainer("small", False)
    with pytest.raises(ValueError, match="config width: 128 in the state, 256 here"):
        small.load_state_dict(_trainer("tiny", True).state_dict())
    with pytest.raises(ValueError, match="config quick_gelu: True in the state, False here"):
        small.load_state_dict(_trainer("small", True).state_dict())
    assert small.opt_step == 0 and float(small.exp_avg.abs().max()) == 0.0


def test_checkpoint_calls_refuse_an_outstanding_exchange():
    """state_dict / load_state_dict between step() calls only: a queued all-reduce of the overlapped gradient exchange (a
    stand-in object here; no collective is needed) makes both raise."""
    tr = _trainer("tiny", True)
    state = tr.state_dict()
    tr._works.append(object())
    with pytest.raises(RuntimeError, match="outstanding"):
        tr.state_dict()
    with pytest.raises(RuntimeError, match="outstanding"):
        tr.load_state_dict(state)
    tr._works.clear()
    tr.load_state_dict(state)

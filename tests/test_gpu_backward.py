"""K4 on the GPU: gradients of the FARE objective (utils_AT.py:317-337) through the engine's backward against torch
autograd over the fp32 oracle tower, for the open_clip and the HF parameter layouts.
Tolerances (the engine multiplies bf16 operands; the reference trains under fp16 autocast):
  * backward alone (same cotangent dL/df fed to both): relative L2 error per tensor <= 3e-2, cosine >= 0.999;
  * end to end (loss.backward()): the TextFARE cotangent 2(f - a)/B is a DIFFERENCE of embeddings, so the forward's
    bf16 error (|df|/|f| ~ 7e-3) is amplified by |f|/|f - a| before it enters the backward: cosine >= 0.995."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _ref_grads(sd, tok, anchor, heads, quick, cotangent=None):
    """fp32 autograd reference. cotangent = None: gradients of the FARE loss; else the vector-Jacobian product."""
    from oracle import leaf_oracle as O
    p = {k: v.detach().clone().cuda().requires_grad_(True) for k, v in sd.items()}
    f = O.encode_text_device(p, tok.cuda(), heads, quick_gelu=quick)
    loss = torch.nn.functional.mse_loss(anchor, f, reduction="none").sum(-1).mean()      # utils_AT.py:321
    if cotangent is None:
        loss.backward()
    else:
        f.backward(cotangent)
    return loss.item(), f.detach(), {k: v.grad for k, v in p.items()}


@pytest.mark.parametrize("name,quick", [("small", False), ("tiny", True)])
def test_backward_matches_autograd(name, quick):
    from leaf_b200 import synth
    from leaf_b200.tower import LeafTextTower
    cfg = synth.TOWERS[name]
    sd = synth.random_tower_state_dict(cfg, seed=11, exact_numpy=True)
    tower = LeafTextTower(sd, heads=cfg.heads, quick_gelu=quick).trainable()
    caps = synth.make_captions(6, seed=5) + synth.make_captions(1, seed=5, kind="dense-77") + ["a", ""]
    tok = tower.tokenizer(caps)
    g = torch.Generator().manual_seed(0)
    with torch.no_grad():
        anchor = tower.encode_text(tok) + 0.3 * torch.randn((len(caps), cfg.embed_dim), generator=g).cuda()
    f = tower.encode_text(tok)
    assert f.requires_grad
    loss = torch.nn.functional.mse_loss(anchor, f, reduction="none").sum(-1).mean()
    loss.backward()
    ref_loss, ref_f, ref = _ref_grads(sd, tok, anchor, cfg.heads, quick)
    assert abs(loss.item() - ref_loss) <= 1e-2 * abs(ref_loss)
    cot = (2.0 * (f.detach() - anchor) / len(caps)).contiguous()            # the cotangent the engine's backward was given
    _, _, vjp = _ref_grads(sd, tok, anchor, cfg.heads, quick, cotangent=cot)

    def err(got, want):
        rel = ((got - want).norm() / want.norm().clamp_min(1e-20)).item()
        return rel, torch.nn.functional.cosine_similarity(got.flatten().double(), want.flatten().double(), dim=0).item()

    for k, safe in tower._names.items():
        got = getattr(tower, safe).grad
        assert got is not None and got.shape == ref[k].shape, k
        rel, cos = err(got, vjp[k])
        assert rel <= 3e-2 and cos >= 0.999, ("backward", k, rel, cos)
        rel, cos = err(got, ref[k])
        assert cos >= 0.995, ("end to end", k, rel, cos)
    # a second backward accumulates (+=) like torch
    f2 = tower.encode_text(tok)
    torch.nn.functional.mse_loss(anchor, f2, reduction="none").sum(-1).mean().backward()
    k0 = "transformer.resblocks.0.mlp.c_fc.weight"
    assert err(getattr(tower, tower._names[k0]).grad, 2 * vjp[k0])[0] <= 3e-2


def test_one_forward_one_backward_is_enforced():
    """The engine keeps ONE saved forward. A backward through an output whose activations were overwritten by a later
    encode_text, a second backward through the same output, or a dfeat of the wrong height must raise - never
    differentiate the wrong activations or read out of bounds."""
    from leaf_b200 import LeafError, synth
    from leaf_b200.tower import LeafTextTower
    tower = LeafTextTower.random("tiny", seed=1).trainable()
    eng = tower.leaf_engine
    tok_a, tok_b = tower.tokenizer(synth.make_captions(4, seed=1)), tower.tokenizer(synth.make_captions(6, seed=2))
    fa = tower.encode_text(tok_a)
    fb = tower.encode_text(tok_b)                          # overwrites fa's activations
    with pytest.raises(LeafError, match="ONE saved forward"):
        fa.sum().backward()
    fb.sum().backward()                                    # the latest forward is still intact
    g1 = tower.flat_grads.clone()
    assert float(g1.abs().max()) > 0
    with pytest.raises(LeafError, match="consumed"):       # its store is gone now
        eng.backward(torch.ones_like(fb), {k: p.grad for k, p in tower.named_tower_parameters()}, eng.last_generation)
    f = eng.forward_train(tok_a)
    grads = {k: p.grad for k, p in tower.named_tower_parameters()}
    with pytest.raises(LeafError, match="rows"):
        eng.backward(torch.ones((3, f.shape[1]), device="cuda"), grads, eng.last_generation)
    with pytest.raises(LeafError):
        eng.backward(torch.ones((4, f.shape[1] + 8), device="cuda"), grads, eng.last_generation)
    eng.backward(torch.ones_like(f), grads, eng.last_generation)
    assert not torch.equal(tower.flat_grads, g1)


def test_train_forward_with_host_lengths_does_not_change_anything():
    """tokenizer(..., with_lengths=True) returns the pooled lengths with its status read; forward_train(host_lengths=...) then
    skips its stream synchronisation (the packed row count sizes the weight-gradient contractions on the host). Same features,
    same gradients as the synchronising path."""
    from leaf_b200 import synth
    from leaf_b200.tower import LeafTextTower
    tower = LeafTextTower.random("small", seed=2).trainable()
    eng = tower.leaf_engine
    caps = synth.make_captions(9, seed=3) + ["", "a"]
    tok, lens = tower.tokenizer(caps, with_lengths=True)
    assert lens == (tok.argmax(dim=-1) + 1).cpu().tolist() and torch.equal(tok, tower.tokenizer(caps))
    grads = []
    for hint in (None, lens):
        tower.zero_grad()
        f = tower.encode_text(tok, host_lengths=hint)
        f.square().sum().backward()
        grads.append((f.detach().clone(), tower.flat_grads.clone()))
    assert torch.equal(grads[0][0], grads[1][0])
    # weight gradients of the 16-48-tile shapes are split-K sums (atomic order): equal to rounding, not to the bit
    assert ((grads[0][1] - grads[1][1]).norm() / grads[0][1].norm()).item() < 1e-5


def test_dependent_launch_changes_no_bit(monkeypatch):
    """The per-layer chain is launched with programmatic dependent launch (a GEMM sets itself up under the tail of the LayerNorm /
    attention kernel before it, csrc/gemm_sm100.cuh pdl_wait): the attack's features must equal, bit for bit, those of an engine
    that launches every kernel ordinarily (LEAF_PDL=0), every time (a kernel that read its predecessor's output before
    pdl_wait() would differ from run to run), and the training forward + backward must agree to the atomics' rounding."""
    from leaf_b200 import synth
    from leaf_b200.tower import LeafTextTower
    sd = synth.random_tower_state_dict(synth.TOWERS["small"], seed=6, device="cuda")
    monkeypatch.setenv("LEAF_PDL", "0")
    plain = LeafTextTower({k: v.clone() for k, v in sd.items()}, heads=4).trainable()
    monkeypatch.delenv("LEAF_PDL")
    chained = LeafTextTower({k: v.clone() for k, v in sd.items()}, heads=4).trainable()
    B, n = 24, 50
    caps = synth.make_captions(B, seed=8)
    rng = np.random.RandomState(2)
    pos = torch.from_numpy(np.stack([rng.randint(0, 2 * len(S) + 1, size=n) for S in caps]).astype(np.int32)).cuda()
    chr_ = torch.from_numpy(np.array(synth.V_DEFAULT, dtype=np.int32)[rng.randint(0, 96, size=(B, n))]).cuda()
    outs = []
    for tower in (plain, chained):
        eng = tower.leaf_engine
        d, o = eng.upload_captions(caps)
        tok, ln, base = eng.expand_tokenize(d, o, B, n, pos, chr_)
        outs.append(eng.encode_tokens(tok, ln, False, base, (B * n, n)))
        for _ in range(5):
            assert torch.equal(outs[-1], eng.encode_tokens(tok, ln, False, base, (B * n, n)))
    assert torch.equal(outs[0], outs[1])
    tok = plain.tokenizer(caps)
    res = []
    for tower in (plain, chained):
        tower.zero_grad()
        f = tower.encode_text(tok)
        f.square().sum().backward()
        res.append((f.detach().clone(), tower.flat_grads.clone()))
    assert torch.equal(res[0][0], res[1][0])
    assert ((res[0][1] - res[1][1]).norm() / res[0][1].norm()).item() < 1e-5


def test_backward_hf_layout():
    from leaf_b200 import synth
    from leaf_b200.engine import LeafEngine
    cfg = synth.TOWERS["small"]
    sd = {k: v.cuda() for k, v in synth.random_tower_state_dict(cfg, seed=4, exact_numpy=True).items()}
    W = cfg.width
    hf = {"text_model.embeddings.token_embedding.weight": sd["token_embedding.weight"],
          "text_model.embeddings.position_embedding.weight": sd["positional_embedding"],
          "text_model.final_layer_norm.weight": sd["ln_final.weight"], "text_model.final_layer_norm.bias": sd["ln_final.bias"],
          "text_projection.weight": sd["text_projection"].T.contiguous()}
    for i in range(cfg.layers):
        p, q = f"transformer.resblocks.{i}.", f"text_model.encoder.layers.{i}."
        for j, nm in enumerate("qkv"):
            hf[q + f"self_attn.{nm}_proj.weight"] = sd[p + "attn.in_proj_weight"][j * W:(j + 1) * W].contiguous()
            hf[q + f"self_attn.{nm}_proj.bias"] = sd[p + "attn.in_proj_bias"][j * W:(j + 1) * W].contiguous()
        for a, b in (("attn.out_proj", "self_attn.out_proj"), ("ln_1", "layer_norm1"), ("ln_2", "layer_norm2"),
                     ("mlp.c_fc", "mlp.fc1"), ("mlp.c_proj", "mlp.fc2")):
            hf[q + b + ".weight"], hf[q + b + ".bias"] = sd[p + a + ".weight"], sd[p + a + ".bias"]
    e1, e2 = LeafEngine(sd, heads=cfg.heads), LeafEngine(hf, heads=cfg.heads)
    tok = e1.tokenize(synth.make_captions(5, seed=1))
    f1, f2 = e1.forward_train(tok), e2.forward_train(tok)
    assert torch.equal(f1, f2)
    # train-mode forward == inference forward (no dropout in the text tower); the two paths round fc1's output at
    # different points (fused GELU epilogue vs saved pre-activation), hence a bf16-level tolerance
    fi = e1.encode_tokens(tok)
    assert (f1 - fi).norm() / fi.norm() < 1e-2
    d = torch.randn_like(f1)
    g1 = {k: torch.zeros_like(v) for k, v in sd.items()}
    g2 = {k: torch.zeros_like(v) for k, v in hf.items()}
    e1.backward(d, g1)
    e2.backward(d, g2)
    assert torch.allclose(g2["text_projection.weight"], g1["text_projection"].T, rtol=1e-3, atol=1e-6)
    for i in range(cfg.layers):
        p, q = f"transformer.resblocks.{i}.", f"text_model.encoder.layers.{i}."
        for j, nm in enumerate("qkv"):
            assert torch.allclose(g2[q + f"self_attn.{nm}_proj.weight"], g1[p + "attn.in_proj_weight"][j * W:(j + 1) * W], rtol=1e-3, atol=1e-6)
            assert torch.allclose(g2[q + f"self_attn.{nm}_proj.bias"], g1[p + "attn.in_proj_bias"][j * W:(j + 1) * W], rtol=1e-3, atol=1e-6)
        assert torch.allclose(g2[q + "mlp.fc1.weight"], g1[p + "mlp.c_fc.weight"], rtol=1e-3, atol=1e-6)


def test_adamw_kernel_matches_torch():
    """leaf_adamw over a flat buffer (no-decay group first) against torch.optim.AdamW with the reference's two parameter
    groups (train_AT_text_only.py:326-341), several steps, with a gradient scale."""
    from leaf_b200.tower import LeafTextTower
    eng = LeafTextTower.random("tiny", seed=0).leaf_engine
    g = torch.Generator(device="cuda").manual_seed(1)
    n, nd = 40960, 1024
    p = torch.randn(n, generator=g, device="cuda")
    ref_a, ref_b = p[:nd].clone().requires_grad_(True), p[nd:].clone().requires_grad_(True)
    lr, b1, b2, eps, wd, scale = 1e-3, 0.9, 0.98, 1e-6, 0.1, 0.5
    opt = torch.optim.AdamW([{"params": [ref_a], "weight_decay": 0.0}, {"params": [ref_b], "weight_decay": wd}], lr=lr,
                            betas=(b1, b2), eps=eps)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    for step in range(1, 6):
        grad = torch.randn(n, generator=g, device="cuda") * (0.1 if step % 2 else 10.0)
        ref_a.grad, ref_b.grad = grad[:nd] * scale, grad[nd:] * scale
        opt.step()
        eng.adamw(p, grad, m, v, n_nodecay=nd, lr=lr, beta1=b1, beta2=b2, eps=eps, weight_decay=wd, step=step, grad_scale=scale)
        want = torch.cat([ref_a.detach(), ref_b.detach()])
        assert torch.allclose(p, want, rtol=1e-5, atol=1e-7), (step, (p - want).abs().max().item())


def test_fare_trainer_matches_a_torch_loop():
    """FareTrainer.step (flat gradient buffer, native AdamW, accumulation, clipping) against the same iteration written as
    the reference writes it (utils_AT.py:291-362) with torch.optim.AdamW on the same engine."""
    import numpy as np
    from leaf_b200 import attack_text_leaf, synth
    from leaf_b200.fare import FareTrainer
    from leaf_b200.tower import LeafTextTower, no_weight_decay
    cfg = synth.TOWERS["small"]
    sd = synth.random_tower_state_dict(cfg, seed=3, exact_numpy=True)
    frozen = LeafTextTower(synth.perturbed_copy(sd, seed=4, std=1e-2, exact_numpy=True), heads=cfg.heads)
    a, b = LeafTextTower(sd, heads=cfg.heads), LeafTextTower(sd, heads=cfg.heads).trainable()
    hp = dict(lr=1e-3, wd=0.05, beta1=0.9, beta2=0.98, eps=1e-6)
    tr = FareTrainer(a, frozen, rho=12, k_adv=1, accum_freq=2, grad_clip_norm=0.5, **hp)
    named = b.named_tower_parameters()
    opt = torch.optim.AdamW([{"params": [p for k, p in named if no_weight_decay(k, p.dim())], "weight_decay": 0.0},
                             {"params": [p for k, p in named if not no_weight_decay(k, p.dim())], "weight_decay": hp["wd"]}],
                            lr=hp["lr"], betas=(hp["beta1"], hp["beta2"]), eps=hp["eps"])
    batches = [synth.make_captions(6, seed=20 + i) for i in range(2)]          # one optimizer step of two micro-batches
    for i, texts in enumerate(batches):
        np.random.seed(100 + i)
        loss_a, adv_a = tr.step(texts)
        np.random.seed(100 + i)
        with torch.no_grad():
            anchors = frozen.encode_text(frozen.tokenizer(texts))
            _, adv_b = attack_text_leaf(b, None, texts, anchors.clone(), "cuda", objective="l2", n=12, k=1)
        feats = b.encode_text(b.tokenizer(adv_b))
        loss_b = torch.nn.functional.mse_loss(anchors, feats, reduction="none").sum(dim=-1).mean()
        (loss_b / 2).backward()
        torch.nn.utils.clip_grad_norm_([p for _, p in named], 0.5, norm_type=2.0)       # after EVERY micro-batch (utils_AT.py:356-357)
        if (i + 1) % 2 == 0:
            opt.step()
            opt.zero_grad()
            b.refresh()
        assert adv_a == adv_b, i
        assert torch.allclose(loss_a, loss_b.detach(), rtol=1e-5), i
    assert tr.opt_step == 1 and float(a.flat_grads.abs().max()) == 0.0
    # AdamW turns every gradient into a step of ~lr whatever its size, and the small gradients are atomic / split-K sums whose
    # order varies run to run: a near-zero gradient may step the other way. So: the update as a whole must agree, and all
    # but a vanishing share of the elements to the usual tolerance.
    sd0 = {k: v.cuda() for k, v in sd.items()}
    for (k, pa), (_, pb) in zip(a.named_tower_parameters(), named):
        upd = (pb - sd0[k]).norm().clamp_min(1e-12)
        assert ((pa - pb).norm() / upd).item() < 2e-2, (k, ((pa - pb).norm() / upd).item())
        bad = ((pa - pb).abs() > 1e-6 + 1e-4 * pb.abs()).float().mean().item()
        assert bad < 1e-3, (k, bad, (pa - pb).abs().max().item())
    assert not torch.equal(a.flat_params, LeafTextTower(sd, heads=cfg.heads).flat_params)      # the update really happened
    # (later steps can legitimately diverge: a 1e-6 difference in a parameter is enough to flip a near-tied candidate)
    tr.step(batches[0]); tr.step(batches[1])
    assert tr.opt_step == 2

"""GPU parity of the text tower (K2) and of the whole attack against the oracle and the golden fixtures generated
from the reference (tests/golden/*, oracle/make_golden.py). Tolerances are BASELINE.json's: embeddings cosine >= 0.999,
TextFARE loss relative error <= 1e-2, selected-candidate agreement >= 99% on non-tied scores."""
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

COS_MIN = 0.999
LOSS_RTOL = 1e-2


def _cos(a, b):
    return torch.nn.functional.cosine_similarity(a.double(), b.double(), dim=-1)


def test_tower_golden_fixtures(golden_dir):
    """Reference CLIP.encode_text outputs (fp32) for the tiny / small towers, gelu and quick_gelu."""
    from leaf_b200 import synth
    from leaf_b200.tower import LeafTextTower
    z = np.load(os.path.join(golden_dir, "tower_golden.npz"))
    tokens = torch.from_numpy(z["tokens"]).cuda()
    for name, quick in (("tiny", False), ("tiny", True), ("small", False)):
        cfg = synth.TOWERS[name]
        sd = synth.random_tower_state_dict(cfg, seed=21, exact_numpy=True)
        tower = LeafTextTower(sd, heads=cfg.heads, quick_gelu=quick)
        tag = f"{name}_{'quick' if quick else 'gelu'}"
        f = tower.encode_text(tokens).cpu()
        want = torch.from_numpy(z[tag])
        assert _cos(f, want).min() >= COS_MIN, (tag, _cos(f, want).min().item())
        assert (f - want).norm() / want.norm() < 1e-2
        fn = tower.encode_text(tokens, normalize=True).cpu()
        assert _cos(fn, torch.from_numpy(z[tag + "_norm"])).min() >= COS_MIN
        assert torch.allclose(fn.norm(dim=-1), torch.ones(fn.shape[0]), atol=1e-5)


def test_tower_on_the_reference_conversion_check_ids(golden_dir):
    """The reference's own tower check input, ids [49406, 1..76] (conversion/convert_2.py:252-253): the row has no
    end-of-text token, so the pooled position is 0 and the engine computes ONE row for it; plus full 77-token rows whose
    maximum sits last / mid-row (positions after it are dead) and a 3-token row."""
    from leaf_b200 import synth
    from leaf_b200.tower import LeafTextTower
    z = np.load(os.path.join(golden_dir, "convert_ids_golden.npz"))
    tokens = torch.from_numpy(z["tokens"]).cuda()
    for name in ("tiny", "small"):
        cfg = synth.TOWERS[name]
        tower = LeafTextTower(synth.random_tower_state_dict(cfg, seed=23, exact_numpy=True), heads=cfg.heads)
        f = tower.encode_text(tokens).cpu()
        assert tower.leaf_engine.last_rows() == 1 + 77 + 39 + 3
        want = torch.from_numpy(z[name])
        assert _cos(f, want).min() >= COS_MIN, (name, _cos(f, want))
        assert (f - want).norm() / want.norm() < 1e-2


def test_tower_hf_layout_binds_identically():
    """The HF CLIPTextModel weight layout (split q/k/v, text_projection.weight = P^T; conversion/convert_2.py:37-99)
    must give the same features as the open_clip layout."""
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
    tok = e1.tokenize(synth.make_captions(16, seed=1))
    assert torch.equal(e1.encode_tokens(tok), e2.encode_tokens(tok))


def test_tower_linear_projection_binds_identically():
    """open_clip's nn.Linear projection (text_projection.weight = P^T, [E, W]) and its parameter form (text_projection = P,
    [W, E]) of the same weights encode to the bit: the engine casts the one, and casts and transposes the other, into the
    same bf16 [E, W] operand. Training binds the .weight form too, and its projection gradient is the transposed one."""
    from leaf_b200 import synth
    from leaf_b200.tower import LeafTextTower
    cfg = synth.TOWERS["small"]
    sd = synth.random_tower_state_dict(cfg, seed=4, exact_numpy=True)
    lin = dict(sd)
    lin["text_projection.weight"] = lin.pop("text_projection").t().contiguous()
    a, b = LeafTextTower(sd, heads=cfg.heads), LeafTextTower(lin, heads=cfg.heads)
    assert b.leaf_engine.embed_dim == cfg.embed_dim
    tok = a.tokenizer(synth.make_captions(16, seed=1))
    for normalize in (False, True):
        assert torch.equal(a.encode_text(tok, normalize=normalize), b.encode_text(tok, normalize=normalize)), normalize
    fa, fb = a.trainable().encode_text(tok), b.trainable().encode_text(tok)
    assert torch.equal(fa, fb)
    d = torch.randn_like(fa)
    (fa * d).sum().backward()
    (fb * d).sum().backward()
    ga, gb = dict(a.named_tower_parameters()), dict(b.named_tower_parameters())
    assert torch.allclose(gb["text_projection.weight"].grad, ga["text_projection"].grad.T, rtol=1e-3, atol=1e-6)
    assert torch.allclose(gb["token_embedding.weight"].grad, ga["token_embedding.weight"].grad, rtol=1e-3, atol=1e-6)


@pytest.mark.parametrize("name", ["ViT-L-14"])
def test_tower_full_width_vs_oracle(name):
    """A full-width tower against the fp32 oracle on a handful of rows (the oracle runs on the host in seconds)."""
    from leaf_b200 import synth
    from leaf_b200.tower import LeafTextTower
    from oracle import leaf_oracle as O
    cfg = synth.TOWERS[name]
    tower = LeafTextTower.random(name, seed=2)
    caps = synth.make_captions(6, seed=2) + synth.make_captions(2, seed=2, kind="dense-77") + ["", "a"]
    tok = tower.tokenizer(caps)
    f = tower.encode_text(tok).cpu()
    sd = {k: v.cpu() for k, v in tower.open_clip_state_dict().items()}
    want = O.encode_text(sd, tok.cpu(), cfg.heads, quick_gelu=cfg.quick_gelu)
    assert torch.equal(tok.cpu(), O.OracleTokenizer()(caps))
    assert _cos(f, want).min() >= COS_MIN, _cos(f, want).min().item()


def test_tower_row_position_invariance():
    """Duplicates must produce bit-identical features wherever they sit in the batch (first-index tie-break)."""
    from leaf_b200 import synth
    from leaf_b200.tower import LeafTextTower
    tower = LeafTextTower.random("small", seed=7)
    caps = synth.make_captions(40, seed=3)
    tok = tower.tokenizer(caps + caps[:7] + ["x"] + caps[5:9])
    f = tower.encode_text(tok)
    assert torch.equal(f[40:47], f[:7]) and torch.equal(f[48:52], f[5:9])


def test_shared_prefix_is_bit_identical():
    """Encoding candidates with shared-prefix reuse (base rows) must equal encoding every row on its own."""
    from leaf_b200 import synth
    from leaf_b200.tower import LeafTextTower
    tower = LeafTextTower.random("small", seed=8)
    eng = tower.leaf_engine
    B, n = 12, 40
    caps = synth.make_captions(B - 2, seed=4) + synth.make_captions(2, seed=4, kind="dense-77")
    rng = np.random.RandomState(1)
    pos = np.stack([rng.randint(0, 2 * len(S) + 1, size=n) for S in caps]).astype(np.int32)
    chr_ = np.array(synth.V_DEFAULT, dtype=np.int32)[rng.randint(0, 96, size=(B, n))]
    d, o = eng.upload_captions(caps)
    tok, ln, base = eng.expand_tokenize(d, o, B, n, torch.from_numpy(pos).cuda(), torch.from_numpy(chr_).cuda())
    shared = eng.encode_tokens(tok, ln, False, base)
    rows_shared = eng.last_rows()
    plain = eng.encode_tokens(tok, ln, False, None)
    rows_plain = eng.last_rows()
    assert torch.equal(shared, plain)
    assert rows_plain == int(ln.sum()) and rows_shared < 0.75 * rows_plain
    # duplicate elimination inside a sample: 'a' / 'A' at the same position tokenize identically
    chr_[:, 1::2] = np.where(chr_[:, 0::2] > 96, chr_[:, 0::2] - 32, chr_[:, 0::2])      # upper-case twins of the even columns
    pos[:, 1::2] = pos[:, 0::2]
    tok, ln, base = eng.expand_tokenize(d, o, B, n, torch.from_numpy(pos).cuda(), torch.from_numpy(chr_).cuda())
    ded = eng.encode_tokens(tok, ln, False, base, (B * n, n))
    rows_ded = eng.last_rows()
    ref = eng.encode_tokens(tok, ln, False, None)
    assert torch.equal(ded, ref)
    assert rows_ded < 0.8 * eng.encode_tokens(tok, ln, False, base).shape[0] * 77 and rows_ded < rows_shared
    # provider trimming: the caption rows are cut down to the prefix some candidate reads; every candidate row keeps its bits
    trimmed = eng.encode_tokens(tok, ln, False, base, (B * n, n), trim=True)
    assert torch.equal(trimmed[:B * n], ded[:B * n]) and eng.last_rows() < rows_ded
    same_pos = np.repeat(pos[:, :1], n, axis=1)                               # phase-2 shape: one position per sample
    tok2, ln2, base2 = eng.expand_tokenize(d, o, B, n, torch.from_numpy(same_pos).cuda(), torch.from_numpy(chr_).cuda())
    full2 = eng.encode_tokens(tok2, ln2, False, base2, (B * n, n))
    rows_full2 = eng.last_rows()
    trim2 = eng.encode_tokens(tok2, ln2, False, base2, (B * n, n), trim=True)
    assert torch.equal(trim2[:B * n], full2[:B * n]) and eng.last_rows() < rows_full2
    # final-layer pruning (out-proj / MLP on the pooled EOS rows only) changes no bit either
    eng.set_prune_last(False)
    try:
        assert torch.equal(eng.encode_tokens(tok, ln, False, base, (B * n, n)), ded)
        assert torch.equal(eng.encode_tokens(tok, ln, True, None), eng.encode_tokens(tok, ln, True, base, (B * n, n)))
    finally:
        eng.set_prune_last(True)


def _golden_attack(golden_dir):
    from leaf_b200 import synth
    g = json.load(open(os.path.join(golden_dir, "attack_golden.json")))
    z = np.load(os.path.join(golden_dir, "attack_golden.npz"))
    cfg = synth.TOWERS[g["tower"]]
    sd = synth.random_tower_state_dict(cfg, seed=g["seed"], exact_numpy=True)
    return g, z, cfg, sd


def test_attack_golden_cases(golden_dir):
    """attack_text_leaf with the reference's numpy seeds against the reference's own outputs."""
    from leaf_b200 import attack_text_leaf
    from leaf_b200.tower import LeafTextTower
    from oracle import leaf_oracle as O
    g, z, cfg, sd = _golden_attack(golden_dir)
    tower = LeafTextTower(sd, heads=cfg.heads)
    otok = O.OracleTokenizer()
    sd_cpu = {k: v.float() for k, v in sd.items()}
    enc = lambda t, normalize: O.encode_text(sd_cpu, t, cfg.heads, normalize=normalize)
    agree = total = 0
    for ci, c in enumerate(g["cases"]):
        anchor = torch.from_numpy(z[f"anchor_{ci}"]).cuda()
        np.random.seed(c["seed"])
        feats, adv = attack_text_leaf(tower, None, c["captions"], anchor.clone(), "cuda", objective=c["objective"], n=c["n"],
                                      k=c["k"])
        assert len(adv) == c["B"] and feats.shape == (c["B"], cfg.embed_dim)
        # replay the oracle with a trace to know which decisions were near-ties
        np.random.seed(c["seed"])
        trace = {}
        _, oadv = O.attack_text_leaf_oracle(enc, otok, c["captions"], torch.from_numpy(z[f"anchor_{ci}"]),
                                            objective=c["objective"], n=c["n"], k=c["k"], trace=trace)
        assert oadv == c["adv"]
        if c["k"] == 1:
            r = trace["rounds"][0]
            for b in range(c["B"]):
                tied = False
                for loss in (r["loss1"][b], r["loss2"][b]):
                    top = torch.topk(loss, 2).values
                    # "non-tied": the runner-up is further than the stated loss tolerance from the winner
                    tied |= bool((top[0] - top[1]).abs() <= LOSS_RTOL * top[0].abs())
                if not tied:
                    total += 1
                    agree += int(adv[b] == c["adv"][b])
                    if adv[b] == c["adv"][b]:
                        want = torch.from_numpy(z[f"feats_{ci}"][b])
                        assert _cos(feats[b].cpu(), want) >= COS_MIN
    assert total >= 10
    assert agree / total >= 0.99, (agree, total)


def test_attack_on_accented_captions_golden(golden_dir):
    """attack_text_leaf on captions with code points up to U+024F against the reference's own runs (attack_latin_golden.*):
    winners must agree wherever the oracle's decisions are clear of the loss tolerance."""
    from leaf_b200 import attack_text_leaf, synth
    from leaf_b200.tower import LeafTextTower
    from oracle import leaf_oracle as O
    g = json.load(open(os.path.join(golden_dir, "attack_latin_golden.json")))
    z = np.load(os.path.join(golden_dir, "attack_latin_golden.npz"))
    cfg = synth.TOWERS[g["tower"]]
    sd = synth.random_tower_state_dict(cfg, seed=g["seed"], exact_numpy=True)
    tower = LeafTextTower(sd, heads=cfg.heads)
    otok = O.OracleTokenizer()
    enc = lambda t, normalize: O.encode_text({k: v.float() for k, v in sd.items()}, t, cfg.heads, normalize=normalize)
    total = agree = 0
    for ci, c in enumerate(g["cases"]):
        anchor = torch.from_numpy(z[f"anchor_{ci}"])
        np.random.seed(c["seed"])
        feats, adv = attack_text_leaf(tower, None, c["captions"], anchor.clone().cuda(), "cuda", n=c["n"], k=c["k"])
        assert torch.equal(tower.encode_text(tower.tokenizer(adv)), feats)
        np.random.seed(c["seed"])
        trace = {}
        _, oadv = O.attack_text_leaf_oracle(enc, otok, c["captions"], anchor, n=c["n"], k=c["k"], trace=trace)
        assert oadv == c["adv"]
        if c["k"] == 1:
            r = trace["rounds"][0]
            for b in range(c["B"]):
                clear = all(bool((torch.topk(l[b], 2).values[0] - torch.topk(l[b], 2).values[1]).abs() > LOSS_RTOL * torch.topk(l[b], 2).values[0].abs())
                            for l in (r["loss1"], r["loss2"]))
                if clear:
                    total += 1
                    agree += int(adv[b] == c["adv"][b])
    assert total >= 5 and agree == total, (agree, total)


def test_attack_full_config_vs_oracle_scores():
    """BASELINE config 1 shape (ViT-L-14 tower, k=1, rho=50) on a reduced batch: every candidate's TextFARE loss
    against the fp32 oracle (rel. err <= 1e-2) and the selected candidates (>= 99 % on non-tied scores)."""
    from leaf_b200 import synth
    from leaf_b200.tower import LeafTextTower
    from oracle import leaf_oracle as O
    cfg = synth.TOWERS["ViT-L-14"]
    B, n = 4, 50
    tower = LeafTextTower.random("ViT-L-14", seed=0)
    sd = {k: v.cpu() for k, v in tower.open_clip_state_dict().items()}
    frozen = synth.perturbed_copy(sd, seed=1, std=1e-3)
    caps = synth.make_captions(B, seed=0)
    otok = O.OracleTokenizer()
    anchor = O.encode_text(frozen, otok(caps), cfg.heads)
    eng = tower.leaf_engine
    rng = np.random.RandomState(0)
    pos = np.stack([rng.choice(range(2 * len(S) + 1), size=n, replace=False) for S in caps]).astype(np.int32)
    strings = [O.edit_sentence(S, int(z), 32) for b, S in enumerate(caps) for z in pos[b]]
    want_feats = O.encode_text(sd, otok(strings), cfg.heads)
    want_loss = O.score(want_feats.view(B, n, -1), anchor)
    d, o = eng.upload_captions(caps)
    tok, ln, base = eng.expand_tokenize(d, o, B, n, torch.from_numpy(pos).cuda(), torch.full((B * n,), 32, dtype=torch.int32).cuda())
    assert torch.equal(tok[:B * n].cpu().long(), otok(strings))
    feats = eng.encode_tokens(tok, ln, False, base)
    best, bf, loss = eng.score(feats, anchor.cuda(), B, n, "l2", want_loss=True)
    assert _cos(feats[:B * n].cpu(), want_feats).min() >= COS_MIN
    rel = ((loss.cpu() - want_loss).abs() / want_loss.abs().clamp_min(1e-12))
    assert rel.max() <= LOSS_RTOL, rel.max().item()
    top = torch.topk(want_loss, 2, dim=-1).values
    nontied = (top[:, 0] - top[:, 1]).abs() > LOSS_RTOL * top[:, 0].abs()
    assert torch.equal(best.cpu().long()[nontied], want_loss.argmax(-1)[nontied])


def test_full_size_properties_vit_h():
    """BASELINE config size (ViT-H-14 text tower, B=128, rho=50): the fp32 oracle cannot run 12 800 ViT-H encodes in
    seconds, so parity at full size rests on size-independent properties: shared-prefix packing is bit-identical to
    encoding every row on its own, duplicate candidates tie exactly, K3's loss/argmax equal torch on the same
    features, and the attack's winners are the argmax of their own phase."""
    from leaf_b200 import synth
    from leaf_b200.tower import LeafTextTower
    tower = LeafTextTower.random("ViT-H-14", seed=0)
    eng = tower.leaf_engine
    B, n = 128, 50
    caps = synth.make_captions(B - 8, seed=0) + synth.make_captions(8, seed=0, kind="dense-77")
    rs = np.random.RandomState(0)
    pos = np.stack([rs.choice(range(2 * len(S) + 1), size=n, replace=False) for S in caps]).astype(np.int32)
    chr_ = np.array(synth.V_DEFAULT, dtype=np.int32)[rs.randint(0, 96, size=(B, n))]
    chr_[:, 7] = chr_[:, 3]                                   # forced duplicates (same position below, same character)
    pos[:, 7] = pos[:, 3]
    d, o = eng.upload_captions(caps)
    tok, ln, base = eng.expand_tokenize(d, o, B, n, torch.from_numpy(pos).cuda(), torch.from_numpy(chr_).cuda())
    assert torch.equal(tok.view(-1, 77)[:B * n].view(B, n, 77)[:, 7], tok[:B * n].view(B, n, 77)[:, 3])
    shared = eng.encode_tokens(tok, ln, False, base, (B * n, n))       # shared prefixes + in-sample duplicates
    rows_shared = eng.last_rows()
    plain = eng.encode_tokens(tok, ln, False, None)
    assert eng.last_rows() == int(ln.sum()) and rows_shared < eng.last_rows()
    assert torch.equal(shared, plain)
    assert torch.isfinite(shared).all()
    f = shared[:B * n].view(B, n, -1)
    assert torch.equal(f[:, 7], f[:, 3])
    anchor = shared[B * n:] + 0.01 * torch.randn((B, f.shape[-1]), generator=torch.Generator().manual_seed(1)).cuda()
    best, bf, loss = eng.score(shared, anchor, B, n, "l2", want_loss=True)
    ref = ((f - anchor.view(B, 1, -1)) ** 2).sum(-1)
    assert torch.allclose(loss, ref, rtol=1e-4, atol=1e-6)
    assert torch.equal(best.long(), loss.argmax(-1))
    assert torch.equal(loss[:, 7], loss[:, 3]) and not (best == 7).any()      # first index wins exact ties
    assert torch.equal(bf, f[torch.arange(B), best.long()])


def test_topk_kernel():
    """leaf_topk: value descending, ties by ascending index; optional second score vector averaged in; prefix length m."""
    from leaf_b200 import synth
    from leaf_b200.tower import LeafTextTower
    eng = LeafTextTower.random("tiny", seed=0).leaf_engine
    g = torch.Generator(device="cuda").manual_seed(3)
    for m_total, m, k in ((1, 1, 1), (97, 96, 10), (5000, 4999, 50), (20000, 19999, 1), (130000, 129999, 1), (130000, 129999, 7)):   # > one launch
        a = torch.randn(m_total, generator=g, device="cuda")
        a[torch.randint(0, m_total, (m_total // 3 + 1,), generator=g, device="cuda")] = 0.25     # plenty of exact ties
        b = torch.randn(m_total, generator=g, device="cuda")
        for sb in (None, b):
            v = a[:m] if sb is None else (a[:m] + sb[:m]) / 2
            order = sorted(range(m), key=lambda i, vv=v.cpu(): (-float(vv[i]), i))[:k]
            idx, val = eng.topk(a, k, m=m, score_b=sb)
            assert idx.cpu().tolist() == order
            assert torch.equal(val.cpu(), v.cpu()[order])


def test_eval_attacks_golden(golden_dir):
    """attack_text_charmer_inference / attack_text_bruteforce on the engine against runs of the reference's own
    functions (utils_attacks.py:395-580; tiny tower, fp32 CPU). The engine scores in bf16, so a decision only has to
    match where the oracle's runner-up is further away than the stated loss tolerance."""
    from leaf_b200 import attack_text_bruteforce, attack_text_charmer_inference, synth
    from leaf_b200.tower import LeafTextTower
    from oracle import leaf_oracle as O
    g = json.load(open(os.path.join(golden_dir, "eval_attack_golden.json")))
    z = np.load(os.path.join(golden_dir, "eval_attack_golden.npz"))
    cfg = synth.TOWERS[g["tower"]]
    sd = synth.random_tower_state_dict(cfg, seed=g["seed"], exact_numpy=True)
    sd2 = synth.random_tower_state_dict(cfg, seed=g["seed2"], exact_numpy=True)
    t1, t2 = LeafTextTower(sd, heads=cfg.heads), LeafTextTower(sd2, heads=cfg.heads)
    otok = O.OracleTokenizer()
    enc = lambda t, normalize: O.encode_text(sd, t, cfg.heads, normalize=normalize)
    enc2 = lambda t, normalize: O.encode_text(sd2, t, cfg.heads, normalize=normalize)
    nv = len(synth.V_DEFAULT)

    def clear(loss, k):           # the k-th and (k+1)-th best scores are further apart than the tolerance
        v = torch.sort(loss, descending=True).values
        return k >= len(v) or bool((v[k - 1] - v[k]).abs() > LOSS_RTOL * v[k - 1].abs())

    total = agree = 0
    for ci, c in enumerate(g["charmer"]):
        a1 = torch.from_numpy(z[f"charmer_anchor_{ci}"])
        a2 = torch.from_numpy(z[f"charmer_anchor2_{ci}"]) if c["two"] else None
        adv, dist_ = attack_text_charmer_inference(t1, None, c["sentence"], a1.clone().cuda(), "cuda", objective=c["objective"],
                                                   n=c["n"], k=c["k"], batch_size=c["batch_size"],
                                                   model_2=t2 if c["two"] else None,
                                                   model_2_anchor_features=a2.clone().cuda() if c["two"] else None)
        assert dist_ == c["dist"]
        trace = {}
        O.attack_text_charmer_oracle(enc, otok, c["sentence"], a1.clone(), objective=c["objective"], n=c["n"], k=c["k"],
                                     batch_size=c["batch_size"], encode_2=enc2 if c["two"] else None,
                                     anchor_2=a2.clone() if c["two"] else None, trace=trace)
        decided = not c["tie_dependent"]
        for r in trace["rounds"]:
            # a clear cut between kept and dropped positions, and a winner clear of every candidate that is not its twin
            l2 = r["loss2"]
            twins = l2 >= l2.max() - 1e-6 * l2.max().abs()
            rest = l2[~twins]
            decided &= clear(r["loss1"], len(r["top"])) and (rest.numel() == 0 or bool(
                (l2.max() - rest.max()).abs() > LOSS_RTOL * l2.max().abs()))
        if decided:
            total += 1
            agree += int(adv == c["adv"])
    for ci, c in enumerate(g["bruteforce"]):
        a1 = torch.from_numpy(z[f"brute_anchor_{ci}"])
        adv, dist_ = attack_text_bruteforce(t1, None, c["sentence"], a1.clone().cuda(), "cuda", batch_size=c["batch_size"],
                                            objective=c["objective"])
        assert dist_ == 1
        trace = {}
        O.attack_text_bruteforce_oracle(enc, otok, c["sentence"], a1.clone(), objective=c["objective"], trace=trace)
        l = trace["loss"]
        rest = l[l < l.max() - 1e-6 * l.max().abs()]
        if bool((l.max() - rest.max()).abs() > LOSS_RTOL * l.max().abs()):
            total += 1
            agree += int(adv == c["adv"])
    assert total >= 6, total
    assert agree == total, (agree, total)


def test_bigg_width_tower_and_rho_sweep():
    """BASELINE config 5's shape in small: the ViT-bigG-14 text-tower WIDTH (1280, 20 heads; a 3-layer copy so the fp32
    oracle finishes in seconds) against the oracle, and attack_text_leaf over rho = 10 .. 200 (rho = 200 > 96 draws
    characters WITH replacement, utils_attacks.py:236): winners are the argmax of their own phase and one edit away."""
    from leaf_b200 import attack_text_leaf, synth
    from leaf_b200.tower import LeafTextTower
    from oracle import leaf_oracle as O
    cfg = synth.TowerCfg("ViT-bigG-14-3L", 1280, 3, 20, 1280)
    tower = LeafTextTower.random(cfg, seed=5)
    caps = synth.make_captions(4, seed=6) + synth.make_captions(1, seed=6, kind="dense-77")
    tok = tower.tokenizer(caps)
    sd = {k: v.cpu() for k, v in tower.open_clip_state_dict().items()}
    want = O.encode_text(sd, tok.cpu(), cfg.heads)
    f = tower.encode_text(tok)
    assert _cos(f.cpu(), want).min() >= COS_MIN
    anchor = (f + 0.05 * torch.randn_like(f)).contiguous()
    for rho in (10, 20, 50, 100, 200):
        np.random.seed(rho)
        feats, adv = attack_text_leaf(tower, None, caps, anchor.clone(), "cuda", objective="l2", n=rho, k=1)
        again = tower.encode_text(tower.tokenizer(adv))
        assert torch.equal(again, feats)                       # the returned features are the winners' own
        for a, c in zip(adv, caps):
            assert abs(len(a) - len(c)) <= 1
        loss_adv = ((feats - anchor) ** 2).sum(-1)
        loss_clean = ((f - anchor) ** 2).sum(-1)
        assert bool((loss_adv >= loss_clean * (1 - LOSS_RTOL)).all()) or rho < 20


def test_bruteforce_on_a_long_caption_is_chunked():
    """attack_text_bruteforce over a 300-character caption: (2*300+1)*96 = 57 696 candidates - more than one leaf_topk launch
    holds and more sequences than one encode pass takes (eval_attacks.MAX_SEQS). The winner must be the first maximal
    candidate of the whole list except the never-scored last one (utils_attacks.py:447), found here by scoring every candidate
    string separately."""
    from leaf_b200 import attack_text_bruteforce, generate_sentence, synth
    from leaf_b200.tower import LeafTextTower
    tower = LeafTextTower.random("tiny", seed=3)
    eng = tower.leaf_engine
    S = " ".join(synth.make_captions(8, seed=31))[:300]
    assert len(S) == 300
    f0 = tower.encode_text(tower.tokenizer([S]))
    anchor = (f0 + 0.05 * torch.randn_like(f0)).contiguous()
    adv, dist_ = attack_text_bruteforce(tower, None, S, anchor.clone(), "cuda", objective="l2")
    V = synth.V_DEFAULT
    cands = [generate_sentence(S, z, c) for z in range(2 * len(S) + 1) for c in V]
    losses = []
    for s in range(0, len(cands), 8192):
        f = tower.encode_text(tower.tokenizer(cands[s:s + 8192]))
        losses.append(((f - anchor) ** 2).sum(-1))
    loss = torch.cat(losses)[:-1]
    best = int(loss.argmax())
    got = cands.index(adv)                                  # first candidate spelling the returned sentence
    assert dist_ == 1 and got <= best and float(loss[got]) >= float(loss[best]) * (1 - 1e-6), (adv, cands[best], float(loss[got]), float(loss[best]))

"""GPU parity tests of the individual kernels, through the C ABI (leaf_b200/lib/libleaf_b200.so).
Floating-point kernels are compared with a plain fp32 torch restatement of the same op on the same bf16-rounded
inputs (tolerances stated per test); the integer tokenizer kernel must equal the oracle bit for bit."""
import json
import os
import random

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from leaf_b200 import synth
    from leaf_b200.tower import LeafTextTower
    tower = LeafTextTower.random("small", seed=3)
    return tower.leaf_engine


def _gelu_ref(x, act):
    return x * torch.sigmoid(1.702 * x) if act == 1 else torch.nn.functional.gelu(x)


@pytest.mark.parametrize("M,N,K", [(128, 256, 64), (128, 256, 256), (300, 384, 128), (77, 64, 128), (1000, 3072, 1024),
                                   (4096, 1024, 4096), (20000, 768, 768), (129, 1280, 5120)])
def test_gemm_epilogues(eng, M, N, K):
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N + K)
    A = (torch.randn((M, K), generator=g, device="cuda") * 0.5).to(torch.bfloat16)
    Bt = (torch.randn((N, K), generator=g, device="cuda") * (K ** -0.5)).to(torch.bfloat16)
    bias = torch.randn((N,), generator=g, device="cuda") * 0.1
    ref = A.float() @ Bt.float().T
    # bf16 store
    C = eng.gemm(A, Bt, None, epilogue=0)
    torch.cuda.synchronize()
    # tolerance: bf16 output rounding (2^-8 relative) on values of magnitude <= ~4
    assert torch.allclose(C.float(), ref, atol=2e-2, rtol=1e-2), (C.float() - ref).abs().max().item()
    # fp32 store + bias: fp32 accumulation order differs from torch only
    C32 = eng.gemm(A, Bt, bias, epilogue=3)
    assert torch.allclose(C32, ref + bias, atol=2e-3, rtol=1e-3), (C32 - ref - bias).abs().max().item()
    # activation epilogues
    for act in (0, 1):
        Ca = eng.gemm(A, Bt, bias, epilogue=1, act=act)
        want = _gelu_ref(ref + bias, act)
        assert torch.allclose(Ca.float(), want, atol=2e-2, rtol=1e-2), (act, (Ca.float() - want).abs().max().item())
    # residual: C += A.Bt^T + bias, rows beyond a device-side row count untouched
    m_live = max(1, M - 37)
    m_dev = torch.tensor([m_live], dtype=torch.int32, device="cuda")
    R = torch.randn((M, N), generator=g, device="cuda")
    R0 = R.clone()
    eng.gemm(A, Bt, bias, epilogue=2, C=R, m_dev=m_dev)
    torch.cuda.synchronize()
    assert torch.allclose(R[:m_live], R0[:m_live] + ref[:m_live] + bias, atol=2e-3, rtol=1e-3)
    assert torch.equal(R[m_live:], R0[m_live:])


@pytest.mark.parametrize("M,N,K", [(256, 256, 64), (256, 256, 4096), (1024, 4096, 4104), (3072, 1024, 6216), (64, 264, 40)])
def test_gemm_mn_major_operands(eng, M, N, K):
    """The K4 products read their operands as they lie: weight gradients C = A^T . B with A [K,M] and B [K,N] (both
    MN-major), data gradients C = A . B with A [M,K] K-major and B [K,N] MN-major. K (the row count of a training batch)
    is arbitrary for the weight-gradient shape: TMA zero-fills the ragged last block."""
    g = torch.Generator(device="cuda").manual_seed(M + N + K)
    At = (torch.randn((K, M), generator=g, device="cuda") * 0.5).to(torch.bfloat16)
    B = (torch.randn((K, N), generator=g, device="cuda") * (K ** -0.5)).to(torch.bfloat16)
    ref = At.float().T @ B.float()
    C = eng.gemm_mn(At, B, None, epilogue=3)
    assert torch.allclose(C, ref, atol=2e-3, rtol=1e-3), (C - ref).abs().max().item()
    acc = torch.randn((M, N), generator=g, device="cuda")                     # += into an fp32 gradient buffer
    acc0 = acc.clone()
    eng.gemm_mn(At, B, None, epilogue=2, C=acc)
    assert torch.allclose(acc, acc0 + ref, atol=2e-3, rtol=1e-3)
    if K % 8 == 0:
        C2 = eng.gemm_mn(At.T.contiguous(), B, None, epilogue=3, a_mn=False)
        assert torch.allclose(C2, ref, atol=2e-3, rtol=1e-3), (C2 - ref).abs().max().item()
        assert torch.equal(C2, C)                                              # same products, same order


def test_gemm_duplicate_rows_bitwise_equal(eng):
    """Numerics must not depend on a row's position (SURVEY.md 7, hard part 5): duplicate candidates must tie."""
    g = torch.Generator(device="cuda").manual_seed(5)
    row = torch.randn((1, 1024), generator=g, device="cuda").to(torch.bfloat16)
    A = row.repeat(777, 1).contiguous()
    Bt = (torch.randn((1024, 1024), generator=g, device="cuda") / 32).to(torch.bfloat16)
    C = eng.gemm(A, Bt, None, epilogue=3)
    assert torch.equal(C, C[0:1].expand_as(C))


def test_gemm_hook_rejects_internal_epilogues(eng):
    """The GEMM hooks take epilogues 0-3 and activations 0-1 (leaf_b200.h). The engine's internal epilogues 4-7 read operands
    these entry points never set (the activation backward's U, the deterministic workspaces), so the hooks refuse them, and
    unknown activation codes, before anything is launched."""
    from leaf_b200 import LeafError
    g = torch.Generator(device="cuda").manual_seed(11)
    A = torch.randn((128, 256), generator=g, device="cuda").to(torch.bfloat16)
    Bt = (torch.randn((256, 256), generator=g, device="cuda") / 16).to(torch.bfloat16)
    C = torch.zeros((128, 256), device="cuda")
    launches = eng.launch_count()
    for epi in range(4, 8):
        with pytest.raises(LeafError, match="epilogue"):
            eng.gemm(A, Bt, None, epilogue=epi, C=C)
    with pytest.raises(LeafError, match="epilogue"):
        eng.gemm_mn(A, Bt[:128], None, epilogue=5, C=torch.zeros((256, 256), device="cuda"))
    with pytest.raises(LeafError, match="activation"):
        eng.gemm(A, Bt, None, epilogue=1, act=2)
    assert eng.launch_count() == launches
    assert torch.equal(C, torch.zeros_like(C))
    ref = A.float() @ Bt.float().T                                            # the engine is still usable
    eng.gemm(A, Bt, None, epilogue=3, C=C)
    assert torch.allclose(C, ref, atol=2e-3, rtol=1e-3), (C - ref).abs().max().item()


def test_layernorm(eng):
    g = torch.Generator(device="cuda").manual_seed(1)
    W = eng.width
    x = torch.randn((1000, W), generator=g, device="cuda") * 3 + 0.5
    gamma = 1 + 0.1 * torch.randn((W,), generator=g, device="cuda")
    beta = 0.1 * torch.randn((W,), generator=g, device="cuda")
    y = eng.test_layernorm(x, gamma, beta)
    ref = torch.nn.functional.layer_norm(x, (W,), gamma, beta, 1e-5)
    # bf16 rounding of the output only
    assert torch.allclose(y.float(), ref, atol=3e-2, rtol=8e-3)


def test_attention_varlen_causal(eng):
    g = torch.Generator(device="cuda").manual_seed(2)
    W, H = eng.width, eng.heads
    lens = [1, 2, 13, 77, 40, 5, 77, 3, 16, 17, 33]
    cu = np.concatenate([[0], np.cumsum(lens)])
    rows = int(cu[-1])
    qkv = torch.randn((rows, 3 * W), generator=g, device="cuda").to(torch.bfloat16)
    meta = torch.tensor([[cu[i], t, 0, cu[i]] for i, t in enumerate(lens)], dtype=torch.int32, device="cuda")
    out = eng.test_attention(qkv, meta).float()

    def ref_attn(q, k, v, first_q):
        t, nq = k.shape[0], q.shape[0]
        q, k, v = (z.float().view(-1, H, 64).transpose(0, 1) for z in (q, k, v))
        mask = torch.full((nq, t), float("-inf"), device="cuda").triu_(1 + first_q)
        return (torch.softmax((q @ k.transpose(-1, -2)) * 0.125 + mask, -1) @ v).transpose(0, 1).reshape(nq, W)

    for i, t in enumerate(lens):
        s = int(cu[i])
        q, k, v = qkv[s:s + t].split(W, dim=-1)
        # tolerance: P is rounded to bf16 before P.V, and the output is stored in bf16
        assert torch.allclose(out[s:s + t], ref_attn(q, k, v, 0), atol=3e-2, rtol=2e-2), i
    # shared prefix: sequence 1 (t = 50) owns positions [p, 50) only and reads positions [0, p) from sequence 0's rows
    for p in (0, 1, 15, 16, 31, 49):
        t0, t1 = 60, 50
        own = t1 - p
        qkv = torch.randn((t0 + own, 3 * W), generator=g, device="cuda").to(torch.bfloat16)
        meta = torch.tensor([[0, t0, 0, 0], [t0, t1, p, 0]], dtype=torch.int32, device="cuda")
        out = eng.test_attention(qkv, meta).float()
        full = torch.cat([qkv[:p], qkv[t0:]])              # the sequence as if it had been computed alone
        q, k, v = full.split(W, dim=-1)
        assert torch.allclose(out[t0:], ref_attn(q[p:], k, v, p), atol=3e-2, rtol=2e-2), p


def test_attention_backward_kernel(eng):
    """K4's tensor-core attention backward against torch autograd of an fp32 attention on the same bf16 inputs: every
    length class (1 row, tile boundaries 16 / 17 / 32 / 33, the full 77)."""
    g = torch.Generator(device="cuda").manual_seed(5)
    W, H = eng.width, eng.heads
    lens = [1, 2, 13, 77, 40, 5, 16, 17, 32, 33, 64, 65]
    cu = np.concatenate([[0], np.cumsum(lens)])
    rows = int(cu[-1])
    qkv = (0.7 * torch.randn((rows, 3 * W), generator=g, device="cuda")).to(torch.bfloat16)
    dout = torch.randn((rows, W), generator=g, device="cuda")
    meta = torch.tensor([[cu[i], t, 0, cu[i]] for i, t in enumerate(lens)], dtype=torch.int32, device="cuda")
    o = eng.test_attention(qkv, meta)
    want = torch.zeros((rows, 3 * W), device="cuda")
    for i, t in enumerate(lens):
        s = int(cu[i])
        x = qkv[s:s + t].float().requires_grad_(True)
        q, k, v = (z.view(t, H, 64).transpose(0, 1) for z in x.split(W, dim=-1))
        mask = torch.full((t, t), float("-inf"), device="cuda").triu_(1)
        out = (torch.softmax((q @ k.transpose(-1, -2)) * 0.125 + mask, -1) @ v).transpose(0, 1).reshape(t, W)
        out.backward(dout[s:s + t])
        want[s:s + t] = x.grad
    for T in (77,):
        got = eng.test_attention_bwd(qkv, o, dout, meta, T).float()
        for name, sl in (("dq", slice(0, W)), ("dk", slice(W, 2 * W)), ("dv", slice(2 * W, 3 * W))):
            a, b = got[:, sl], want[:, sl]
            rel = ((a - b).norm() / b.norm()).item()
            # P, dS and dO enter the products as bf16 and the result is stored as bf16
            assert rel < 1.5e-2, (name, T, rel)
            assert torch.allclose(a, b, atol=6e-2, rtol=6e-2), (name, T, (a - b).abs().max().item())


def test_score_argmax(eng):
    g = torch.Generator(device="cuda").manual_seed(3)
    E = eng.embed_dim
    B, n = 9, 50
    feats = torch.randn((B * n, E), generator=g, device="cuda")
    feats[7] = feats[3]                       # exact tie inside sample 0 -> first index must win
    anchor = torch.randn((B, E), generator=g, device="cuda")
    for obj in ("l2", "negl2", "sim", "dissim"):
        best, bf, loss = eng.score(feats, anchor, B, n, obj, want_loss=True)
        f = feats.view(B, n, E)
        if obj in ("l2", "negl2"):
            ref = ((f - anchor.view(B, 1, E)) ** 2).sum(-1)
        else:
            ref = (f @ anchor.view(B, E, 1)).squeeze(-1)
        if obj in ("negl2", "dissim"):
            ref = -ref
        assert torch.allclose(loss, ref, rtol=1e-4, atol=1e-4)
        assert torch.equal(best.long(), torch.argmax(loss, dim=-1))
        assert torch.equal(bf, f[torch.arange(B), best.long()])
    f = feats.clone()
    f[3] = f[7] = anchor[0] + 100.0
    best, _, _ = eng.score(f, anchor, B, n, "l2")
    assert int(best[0]) == 3


# ----------------------------------------------------------------------------------------------------------------
# K1: bit-exact against the oracle / reference goldens
# ----------------------------------------------------------------------------------------------------------------
def _k1(eng, caps, n=0, pos=None, chr_=None, sel=None, valid=None):
    d, o = eng.upload_captions(caps)
    t = lambda a, dt: None if a is None else torch.as_tensor(np.ascontiguousarray(a), dtype=dt).cuda()
    tok, ln, base = eng.expand_tokenize(d, o, len(caps), n, t(pos, torch.int32), t(chr_, torch.int32), t(sel, torch.int32),
                                        t(valid, torch.uint8))
    torch.cuda.synchronize()
    R = len(caps) * max(n, 1)
    if n > 0:      # the B unedited captions follow the candidates, and every candidate names its caption row
        from oracle import leaf_oracle as O
        assert tok.shape[0] == R + len(caps)
        assert torch.equal(tok[R:].cpu().long(), O.OracleTokenizer()(list(caps)))
        assert base[:R].cpu().tolist() == [R + r // n for r in range(R)] and (base[R:] == -1).all()
    return tok[:R].cpu().numpy(), ln[:R].cpu().numpy()


def test_k1_golden_strings(eng, golden_dir):
    from oracle import leaf_oracle as O
    import html
    g = json.load(open(os.path.join(golden_dir, "tokenizer_golden.json")))
    texts = [t for t, _ in g["encode"] if len(t) <= 1000 and all(ord(c) < 128 for c in t)
             and all(ord(c) <= 0xFF for c in html.unescape(t) + html.unescape(html.unescape(t)))]
    assert len(texts) > 2000
    want = O.OracleTokenizer()(texts).numpy()
    tok, ln = _k1(eng, texts)
    eng._status.zero_()
    assert (tok == want).all()
    assert (ln == want.argmax(1) + 1).all()
    tok, ln = _k1(eng, g["rows_in"])
    assert tok.tolist() == g["rows"]


def test_k1_latin1_utf8_captions(eng, golden_dir):
    """Accented captions (UTF-8, code points <= U+024F) on the device: the reference's SimpleTokenizer rows, attack-shaped
    edits with positions counted in code points, the whole attack on such captions, and LeafError beyond the domain."""
    from leaf_b200 import LeafError, attack_text_leaf
    g = json.load(open(os.path.join(golden_dir, "tokenizer_latin1_golden.json")))
    assert eng.tokenize(g["rows_in"]).cpu().tolist() == g["rows"]
    by_s = {}
    for S, z, c, out, ids in g["edits"]:
        by_s.setdefault(S, []).append((z, c, ids))
    for S, cases in by_s.items():
        pos = np.array([[c[0] for c in cases]], dtype=np.int32)
        chr_ = np.array([[c[1] for c in cases]], dtype=np.int32)
        tok, ln = _k1(eng, [S], len(cases), pos, chr_)
        for j, (_, _, ids) in enumerate(cases):
            want = ([49406] + ids + [49407])[:77]
            want[-1] = 49407
            assert tok[j, :len(want)].tolist() == want and not tok[j, len(want):].any(), (S, cases[j])
    eng._status.zero_()
    caps = g["rows_in"][:6]
    anchor = eng.encode_tokens(eng.tokenize(caps)) + 0.1
    np.random.seed(3)
    feats, adv = attack_text_leaf(eng, None, caps, anchor, "cuda", n=12, k=2)
    assert all(abs(len(a) - len(c)) <= 2 for a, c in zip(adv, caps)) and adv != caps
    assert torch.equal(eng.encode_tokens(eng.tokenize(adv)), feats)
    for bad in ("na\u00efve \u0250", "emoji \U0001F600"):
        with pytest.raises(LeafError, match="U\\+024F"):
            eng.tokenize([bad])
    with pytest.raises(LeafError, match="domain"):
        eng.tokenize(["\u0130stanbul"])                                           # str.lower() leaves the domain
    with pytest.raises(LeafError, match="domain"):
        eng.tokenize(["mojibake Ã©"])
    eng._status.zero_()


def test_k1_long_captions(eng):
    """Captions of 1000-3560 bytes switch the tokenizer kernel to its long-text variant (sticky per engine); rows equal the oracle's
    and the CPU-compiled core's, the attack runs on them, and longer captions raise."""
    from leaf_b200 import LeafError, attack_text_leaf, synth
    from leaf_b200.tower import LeafTextTower
    from oracle import leaf_oracle as O
    from tests import k1_harness as H
    e = LeafTextTower.random("tiny", seed=2).leaf_engine                     # its own engine: the switch is sticky
    caps = [" ".join(synth.make_captions(40, seed=s))[:L] for s, L in ((1, 1500), (2, 2600), (3, 3560))] + ["short one", "caf\u00e9 " * 500]
    assert torch.equal(e.tokenize(caps).cpu(), O.OracleTokenizer()(caps))
    rng = np.random.RandomState(0)
    n = 16
    pos = np.stack([rng.randint(0, 2 * len(S) + 1, size=n) for S in caps]).astype(np.int32)
    chr_ = np.array(synth.V_DEFAULT, dtype=np.int32)[rng.randint(0, 96, size=(len(caps), n))]
    tok, ln = _k1(e, caps, n, pos, chr_)
    htok, hln, _ = H.expand_tokenize(caps, n, pos, chr_)
    assert (tok == htok).all() and (ln == hln).all()
    anchor = e.encode_tokens(e.tokenize(caps)) + 0.1
    np.random.seed(1)
    feats, adv = attack_text_leaf(e, None, caps, anchor, "cuda", n=8, k=1)
    assert torch.equal(e.encode_tokens(e.tokenize(adv)), feats) and all(abs(len(a) - len(c)) <= 1 for a, c in zip(adv, caps))
    with pytest.raises(LeafError, match="longer"):
        e.tokenize(["z" * 3561])


def test_k1_candidates_bit_exact(eng):
    from leaf_b200 import synth
    from oracle import leaf_oracle as O
    rng = random.Random(5)
    otok = O.OracleTokenizer()
    V = synth.V_DEFAULT
    for kind, B, n in (("typical", 32, 50), ("dense-77", 6, 50), ("short", 12, 120)):
        caps = synth.make_captions(B, seed=9, kind=kind)
        pos = np.array([[rng.randint(0, 2 * len(S)) for _ in range(n)] for S in caps], dtype=np.int32)
        chr_ = np.array([[V[rng.randrange(len(V))] for _ in range(n)] for _ in caps], dtype=np.int32)
        valid = np.ones((B, n), dtype=np.uint8)
        valid[:, 5::7] = 0
        tok, ln = _k1(eng, caps, n, pos, chr_, valid=valid)
        strings = [O.edit_sentence(S, int(pos[b, j]), int(chr_[b, j])) if valid[b, j] else S
                   for b, S in enumerate(caps) for j in range(n)]
        want = otok(strings).numpy()
        assert (tok == want).all(), kind
        assert (ln == want.argmax(1) + 1).all()
        sel = np.array([rng.randrange(n) for _ in caps], dtype=np.int32)
        tok, ln = _k1(eng, caps, n, pos, chr_, sel=sel)
        strings = [O.edit_sentence(S, int(pos[b, sel[b]]), int(chr_[b, j])) for b, S in enumerate(caps) for j in range(n)]
        assert (tok == otok(strings).numpy()).all(), kind
    eng._status.zero_()


def test_k1_flags_out_of_domain(eng):
    from leaf_b200 import LeafError
    from oracle import leaf_oracle as O
    assert torch.equal(eng.tokenize(["café"]).cpu(), O.OracleTokenizer()(["café"]))       # Latin-1 / Latin Extended is inside the domain now
    with pytest.raises(LeafError):
        eng.tokenize(["caf\u00e9 \u0250"])                                                 # U+0250 is not
    with pytest.raises(LeafError):
        eng.tokenize(["x &lambda; y"])
    with pytest.raises(LeafError):
        eng.tokenize(["x &amp;amp;lt; y"])                                                 # ftfy would unescape a third level
    assert eng.tokenize(["x &lt; y"]).shape == (1, 77)


def test_k1_matches_cpu_compiled_core_at_full_size(eng):
    """BASELINE config size (B=128, n=50): the device kernel against the same scalar core compiled for the CPU."""
    from leaf_b200 import synth
    from tests import k1_harness as H
    rng = np.random.RandomState(0)
    caps = synth.make_captions(128, seed=0, kind="typical")
    n = 50
    pos = np.stack([rng.randint(0, 2 * len(S) + 1, size=n) for S in caps]).astype(np.int32)
    chr_ = np.array(synth.V_DEFAULT, dtype=np.int32)[rng.randint(0, 96, size=(128, n))]
    tok, ln = _k1(eng, caps, n, pos, chr_)
    htok, hln, _ = H.expand_tokenize(caps, n, pos, chr_)
    assert (tok == htok).all() and (ln == hln).all()
    eng._status.zero_()


def test_constrain_mask_matches_oracle(eng):
    """leaf_constrain_mask (thread per sentence) against the oracle's restatement of valid_sentence_batched
    (utils_attacks.py:110-143 over nltk.word_tokenize, oracle/nltk_restate.py), both phases' candidate forms, and the
    CPU-compiled core at the full attack size."""
    from leaf_b200 import synth
    from oracle import leaf_oracle as O
    from oracle import nltk_restate as N
    from tests import k1_harness as H
    from tests.test_constrain_cpu import ABBREV, _texts, _word_list
    words = _word_list()
    eng.load_words(words, ABBREV)
    H.load_words(words, ABBREV)
    W, A = frozenset(words), frozenset(ABBREV)
    V = np.asarray(synth.V_DEFAULT, dtype=np.int32)
    caps = synth.make_captions(10, seed=3) + ["a photo of a cat's toy, isn't it? yes. the dog (brown) can't stop.",
                                               'he said "hello there." then left -- cannot go', "mr. smith's dog & cat: a,b"] \
        + [t for t in _texts(7, 40) if t.isascii() and len(t) > 0][:20]
    B, n = len(caps), 50
    rs = np.random.RandomState(1)
    pos = np.stack([rs.randint(0, 2 * len(S) + 1, size=n) for S in caps]).astype(np.int32)
    chr_ = V[rs.randint(0, len(V), size=(B, n))]
    d, o = eng.upload_captions(caps)
    pos_d, chr_d = torch.from_numpy(pos).cuda(), torch.from_numpy(chr_).cuda()
    valid, counts = eng.constrain_mask(d, o, B, n, pos_d, chr_d, want_counts=True)
    eng.check_status()
    SS = [[O.edit_sentence(S, int(z), int(c)) for z, c in zip(pos[b], chr_[b])] for b, S in enumerate(caps)]
    want = np.asarray(N.valid_sentence_batched(caps, SS, W, A), dtype=np.uint8)
    assert np.array_equal(valid.cpu().numpy(), want)
    assert counts[B * n:].cpu().tolist() == [N.count_dictionary_words(S, W, A) for S in caps]
    sel = torch.from_numpy(rs.randint(0, n, size=B).astype(np.int32)).cuda()
    valid2 = eng.constrain_mask(d, o, B, n, pos_d, chr_d, sel)
    SS2 = [[O.edit_sentence(S, int(pos[b, int(sel[b])]), int(c)) for c in chr_[b]] for b, S in enumerate(caps)]
    assert np.array_equal(valid2.cpu().numpy(), np.asarray(N.valid_sentence_batched(caps, SS2, W, A), dtype=np.uint8))
    # the mask feeds leaf_expand_tokenize: invalid candidates come back as the unedited caption's row
    tok, ln, base = eng.expand_tokenize(d, o, B, n, pos=pos_d, chr_=chr_d, valid=valid)
    inv = (valid.view(-1) == 0).nonzero().flatten()
    assert inv.numel() > 0 and torch.equal(tok[inv], tok[B * n + inv // n])
    # full attack size against the CPU-compiled core
    caps = synth.make_captions(128, seed=11)
    B = 128
    pos = np.stack([rs.randint(0, 2 * len(S) + 1, size=n) for S in caps]).astype(np.int32)
    chr_ = V[rs.randint(0, len(V), size=(B, n))]
    d, o = eng.upload_captions(caps)
    _, counts = eng.constrain_mask(d, o, B, n, torch.from_numpy(pos).cuda(), torch.from_numpy(chr_).cuda(), want_counts=True)
    hc, flags = H.constrain_counts(caps, n, pos, chr_)
    assert flags == 0 and np.array_equal(counts.cpu().numpy(), hc)


def test_constrain_kernel_counts_nltk_published_vectors(eng):
    """leaf_constrain_mask on the word_tokenize vectors NLTK itself publishes (tests/golden/nltk_published_vectors.json): with the
    published tokens as the dictionary the device count is the number of distinct published tokens, with the glued
    whitespace forms as the dictionary it is 0 (same check as tests/test_constrain_cpu.py runs on the CPU-compiled core)."""
    from tests.test_constrain_cpu import published_count_cases
    cases = published_count_cases()
    assert len(cases) >= 15
    pos = torch.zeros((1, 1), dtype=torch.int32, device="cuda")
    chr_ = torch.full((1, 1), -1, dtype=torch.int32, device="cuda")
    for text, abbrev, want, glued in cases:
        d, o = eng.upload_captions([text])
        eng.load_words(want, abbrev)
        _, counts = eng.constrain_mask(d, o, 1, 1, pos, chr_, want_counts=True)
        assert counts.cpu().tolist() == [len(want), len(want)], (text, counts.cpu().tolist(), want)
        if glued:
            eng.load_words(glued, abbrev)
            _, counts = eng.constrain_mask(d, o, 1, 1, pos, chr_, want_counts=True)
            assert counts.cpu().tolist() == [0, 0], (text, glued)
    eng.check_status()


def test_hf_tokenizer_mode_and_hf_shaped_rows(eng, golden_dir):
    """HF wire compatibility (SURVEY.md 8f item 4): token ids of transformers' CLIPTokenizer, the tokenizer_wrapper layout
    (padded to the longest row with the pad id), and the forward on such rows with HF's first-EOS pooling."""
    g = json.load(open(os.path.join(golden_dir, "hf_tokenizer_golden.json")))
    eng.set_tokenizer_mode(True)
    try:
        for batch, rows in g["wrapped"]:
            got = eng.tokenize_hf(batch, pad_id=g["pad_id"])
            assert got.cpu().tolist() == rows
        texts = [s for s, _ in g["encode"] if len(s) <= 1000][:300]
        tok = eng.tokenize(texts)
        for i, (s, ids) in enumerate([(s, ids) for s, ids in g["encode"] if len(s) <= 1000][:300]):
            want = ids if len(ids) <= 77 else ids[:76] + [49407]
            assert tok[i, :len(want)].cpu().tolist() == want, s
        # forward on HF-shaped rows == forward on the engine's own 77-slot rows
        batch = g["wrapped"][1][0]
        hf_rows = eng.tokenize_hf(batch, pad_id=g["pad_id"])
        assert hf_rows.shape[1] < 77
        f_hf = eng.encode_hf_tokens(hf_rows, eos_token_id=g["eos_id"])
        f = eng.encode_tokens(eng.tokenize(batch))
        assert torch.equal(f_hf, f)
        f_pad0 = eng.encode_hf_tokens(torch.where(hf_rows == g["pad_id"], torch.zeros_like(hf_rows), hf_rows).where(
            torch.arange(hf_rows.shape[1], device="cuda").view(1, -1) >= (hf_rows == g["eos_id"]).int().argmax(1, keepdim=True) + 1,
            hf_rows), eos_token_id=g["eos_id"])
        assert torch.equal(f_pad0, f)                                   # the pad id after the EOS never matters
    finally:
        eng.set_tokenizer_mode(False)

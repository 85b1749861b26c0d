"""Host-side wrapper of the native engine: owns a leaf_handle_t, binds a text tower's live parameters and exposes
the three duck-typed pieces of the reference's seam (SURVEY.md 8b):

    tokenizer(list[str]) -> LongTensor[N,77]          /root/reference/src/open_clip/tokenizer.py:226-265
    model.encode_text(tokens, normalize) -> [N,E]     /root/reference/src/open_clip/model.py:269-284
    attack_text_leaf(...)                              /root/reference/utils_attacks.py:297-393  (leaf_b200/attack.py)

PyTorch is used for device memory, streams and (elsewhere) torch.distributed only; all compute is in
leaf_b200/lib/libleaf_b200.so, and nothing here runs without it and a B200.
"""
from __future__ import annotations

import contextlib
import ctypes
import os
from dataclasses import dataclass

import numpy as np
import torch

from . import _native
from ._native import BACKWARD_HOOK, LAYER_PARAMS, LAYER_PREFIX, TOWER_PARAMS, LeafCfg, LeafError, LeafLayerPtrs, LeafWeightPtrs, check

HERE = os.path.dirname(os.path.abspath(__file__))
MERGES_BIN = os.path.join(HERE, "data", "clip_bpe_merges.bin")

CONTEXT_LENGTH = 77
OBJECTIVES = {"l2": 0, "negl2": 1, "sim": 2, "dissim": 3}
STATUS_ENTITY_DOMAIN, STATUS_NON_ASCII, STATUS_TOO_LONG = 1, 2, 4
MAX_CAPTION_BYTES = 1000            # the tokenizer kernel's default variant; up to MAX_CAPTION_BYTES_LONG with its long-text variant
MAX_CAPTION_BYTES_LONG = 3560
MAX_CODE_POINT = 0x24F               # csrc/k1_core.cuh: ASCII, Latin-1 Supplement, Latin Extended-A / -B


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


@dataclass
class TowerParams:
    """A text tower's tensors (the parameter dict's own objects) keyed by the ABI field that carries each (TOWER_PARAMS / LAYER_PARAMS)."""
    layout: str                        # "open_clip" or "hf"
    top: dict
    layers: list                       # per layer, the fields its naming has
    projection_is_ew: int              # 1: text_projection is [E, W] (HF, open_clip's nn.Linear); 0: open_clip's [W, E]
    projection_synthesised: bool = False

    def tensors(self) -> list:
        """The tensors of the dict the view was read from: every field but a synthesised projection, None entries left out."""
        top = [t for f, t in self.top.items() if f != "text_projection" or not self.projection_synthesised]
        return [t for t in top + [t for l in self.layers for t in l.values()] if t is not None]


def _canon_state(params: dict) -> TowerParams:
    """The TowerParams of a dict in open_clip (bare or `text.`-prefixed) or HF (CLIPTextModel(WithProjection), CLIPModel) naming."""
    hf_tok = TOWER_PARAMS["token_embedding"][1]
    pre = next((k[: -len(hf_tok)] for k in params if k.endswith(hf_tok)), None)      # "text_model." or "...text_model."
    col = int(pre is not None)
    if col:
        root = pre.removesuffix("text_model.")                         # HF keeps the projection beside text_model
    else:
        pre = root = "text." if "text.token_embedding.weight" in params else ""
        if (pre + "token_embedding.weight") not in params:
            raise LeafError("unrecognised parameter naming: expected open_clip (token_embedding.weight / "
                            "text.token_embedding.weight) or HF CLIPTextModel keys")
    top = {f: params[pre + n[col]] for f, n in TOWER_PARAMS.items() if f != "text_projection"}
    v = TowerParams(("open_clip", "hf")[col], top, [], projection_is_ew=col)
    proj = root + TOWER_PARAMS["text_projection"][col]
    if proj in params:
        top["text_projection"] = params[proj]
    elif col:                          # CLIPTextModel: the reference reads .pooler_output (utils_attacks.py:49-53) = identity head
        top["text_projection"] = torch.eye(top["token_embedding"].shape[1], dtype=torch.float32, device=top["token_embedding"].device)
        v.projection_synthesised = True
    else:                              # open_clip's nn.Linear projection: an [E, W] weight, like HF's
        top["text_projection"], v.projection_is_ew = params[proj + ".weight"], 1
    layer, names = pre + LAYER_PREFIX[col], {f: n[col] for f, n in LAYER_PARAMS.items() if n[col]}
    while (p := layer.format(len(v.layers))) + names["ln1_w"] in params:
        v.layers.append({f: params[p + n] for f, n in names.items()})
    return v


class LeafEngine:
    """One engine = one text tower on one GPU. `params` is a dict name -> CUDA fp32 tensor (e.g.
    dict(model.named_parameters()) or a state_dict) in open_clip or HF naming; the tensors stay owned by the
    caller and are read in place (call refresh_weights() after every optimizer step)."""

    def __init__(self, params: dict, heads: int, quick_gelu: bool = False, ln_eps: float = 1e-5, max_seqs: int = 0):
        if not torch.cuda.is_available():
            raise LeafError("leaf_b200 needs a CUDA device (sm_100a); there is no CPU path")
        self._lib = _native.lib()
        self._params = v = _canon_state(params)
        self.width = int(v.top["token_embedding"].shape[1])
        self.layers = len(v.layers)
        self.heads = int(heads)
        self.quick_gelu, self.ln_eps = bool(quick_gelu), float(ln_eps)
        self.embed_dim = int(v.top["text_projection"].shape[0 if v.projection_is_ew else 1])
        self.device = v.top["token_embedding"].device
        self._check_tensors()
        cfg = LeafCfg(self.width, self.layers, self.heads, self.embed_dim, 1 if quick_gelu else 0, ln_eps)
        self._h = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            check(self._lib.leaf_create(ctypes.byref(cfg), ctypes.byref(self._h)))
            pairs = np.fromfile(MERGES_BIN, dtype="<u4")
            check(self._lib.leaf_load_bpe(self._h, pairs.ctypes.data_as(ctypes.c_void_p), len(pairs)))
            self._bind()
        self._status = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.deterministic = False
        self.has_words = False
        self.max_seqs = 0
        self._caption_limit = MAX_CAPTION_BYTES
        if max_seqs:
            self.reserve(max_seqs)

    # ---- lifetime ----------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.leaf_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check_tensors(self):
        if not self._params.layers:
            raise LeafError("no transformer layers found in the parameter dict")
        for t in self._params.tensors():
            if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
                raise LeafError("tower parameters must be contiguous fp32 CUDA tensors")
            if t.data_ptr() % 16:
                raise LeafError("tower parameters must be 16-byte aligned")
        if self.width != self.heads * 64:
            raise LeafError(f"head_dim must be 64 (width {self.width}, heads {self.heads})")

    def _make_ptrs(self, v: TowerParams):
        """leaf_weight_ptrs_t over a TowerParams (fields it does not hold, and None entries, become NULL)."""
        ptrs = lambda d: {f: None if t is None else t.data_ptr() for f, t in d.items()}
        arr = (LeafLayerPtrs * self.layers)(*(LeafLayerPtrs(**ptrs(l)) for l in v.layers))
        wp = LeafWeightPtrs(**ptrs(v.top), projection_is_ew=v.projection_is_ew, layers=arr)
        return arr, wp

    def _bind(self):
        self._keep = self._make_ptrs(self._params)
        check(self._lib.leaf_bind_weights(self._h, ctypes.byref(self._keep[1]), _stream()))

    def refresh_weights(self):
        """Re-cast the bf16 operand copies from the live fp32 parameters (after optimizer.step())."""
        with torch.cuda.device(self.device):
            check(self._lib.leaf_refresh_weights(self._h, _stream()))

    def reserve(self, max_seqs: int):
        if max_seqs > self.max_seqs:
            with torch.cuda.device(self.device):
                check(self._lib.leaf_reserve(self._h, int(max_seqs)))
            self.max_seqs = int(max_seqs)

    # ---- K1 ----------------------------------------------------------------------------------------------
    @staticmethod
    def pack_captions(sentences):
        """list[str] -> (uint8 caption bytes back to back, int32 [B+1] BYTE offsets). Captions travel as UTF-8; the kernel's
        domain is code points <= U+024F (ASCII, Latin-1 Supplement, Latin Extended-A / -B; csrc/k1_core.cuh), checked here for a clear message and
        again on the device. The buffer tail is padded so the kernel's 16-byte loads never leave the allocation."""
        blobs = []
        for s in sentences:
            if not s.isascii() and max(map(ord, s)) > MAX_CODE_POINT:
                bad = next(c for c in s if ord(c) > MAX_CODE_POINT)
                raise LeafError(f"caption outside the tokenizer kernel's domain (code points <= U+{MAX_CODE_POINT:04X}): U+{ord(bad):04X} in {s!r}")
            b = s.encode("utf-8")
            if len(b) > MAX_CAPTION_BYTES_LONG:
                raise LeafError(f"caption longer than {MAX_CAPTION_BYTES_LONG} bytes")
            blobs.append(b)
        off = np.zeros(len(blobs) + 1, dtype=np.int32)
        off[1:] = np.cumsum([len(b) for b in blobs])
        data = np.frombuffer(b"".join(blobs) + b"\0" * 32, dtype=np.uint8)
        return data, off

    def upload_captions(self, sentences):
        data, off = self.pack_captions(sentences)
        longest = int(np.diff(off).max()) if len(off) > 1 else 0
        if longest > self._caption_limit:                   # sticky: the long-text kernel variant handles short captions too
            self._caption_limit = MAX_CAPTION_BYTES_LONG
            check(self._lib.leaf_set_max_caption_bytes(self._h, MAX_CAPTION_BYTES_LONG))
        d = torch.from_numpy(data.copy()).pin_memory().to(self.device, non_blocking=True)
        o = torch.from_numpy(off).pin_memory().to(self.device, non_blocking=True)
        return d, o

    def expand_tokenize(self, caps_dev, off_dev, B, n, pos=None, chr_=None, sel=None, valid=None):
        """leaf_expand_tokenize on device tensors; returns (tokens int32 [R,77], lengths int32 [R], base int32 [R]).
        n == 0: R = B (the captions). n > 0: R = B*n + B, the candidates followed by the B unedited captions; base[r]
        names the caption row of candidate r (shared-prefix reuse in encode_tokens), -1 for the caption rows."""
        R = B * n + B if n > 0 else B
        tok = torch.empty((R, CONTEXT_LENGTH), dtype=torch.int32, device=self.device)
        ln = torch.empty((R,), dtype=torch.int32, device=self.device)
        base = torch.empty((R,), dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            check(self._lib.leaf_expand_tokenize(self._h, _ptr(caps_dev), _ptr(off_dev), B, n, _ptr(pos), _ptr(chr_), _ptr(sel),
                                                 _ptr(valid), _ptr(tok), _ptr(ln), _ptr(base), _ptr(self._status), _stream()))
        return tok, ln, base

    # ---- --constrain on the device ----------------------------------------------------------------------------------
    @staticmethod
    def _pack_words(words):
        blobs = [w.encode("ascii") for w in words if w.isascii()]
        off = np.zeros(len(blobs) + 1, dtype=np.int32)
        off[1:] = np.cumsum([len(b) for b in blobs])
        return np.frombuffer(b"".join(blobs) + b"\0", dtype=np.uint8).copy(), off, len(blobs)

    def load_words(self, words, abbrev=()):
        """The dictionary W of the reference's filter (utils_attacks.py:125: set(nltk.corpus.words.words())) and,
        optionally, Punkt's abbreviation types (nltk ... PunktSentenceTokenizer._params.abbrev_types). After this,
        attack_text_leaf(..., constrain=True) computes the validity masks on the device."""
        wb, wo, nw = self._pack_words(words)
        ab, ao, na = self._pack_words(abbrev)
        p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        with torch.cuda.device(self.device):
            check(self._lib.leaf_load_words(self._h, p(wb), p(wo), nw, p(ab) if na else None, p(ao) if na else None, na))
        self.has_words = True

    def constrain_mask(self, caps_dev, off_dev, B, n, pos, chr_, sel=None, want_counts=False):
        """valid uint8 [B,n] (and the int32 dictionary-word counts [B*n+B]) for the candidates of expand_tokenize."""
        valid = torch.empty((B, n), dtype=torch.uint8, device=self.device)
        counts = torch.empty((B * n + B,), dtype=torch.int32, device=self.device) if want_counts else None
        with torch.cuda.device(self.device):
            check(self._lib.leaf_constrain_mask(self._h, _ptr(caps_dev), _ptr(off_dev), B, n, _ptr(pos), _ptr(chr_), _ptr(sel),
                                                _ptr(valid), _ptr(counts), _ptr(self._status), _stream()))
        return (valid, counts) if want_counts else valid

    def check_status(self):
        """Synchronising read of the tokenizer status flags; raises on inputs outside the kernel's closed domain."""
        st = int(self._status.item())
        if st:
            self._status.zero_()
            what = [m for bit, m in ((1, "an html entity expanded outside U+0000..U+024F, or entity text ftfy would unescape differently "
                                         "(third nesting level / ALL-CAPS name)"),
                                     (2, "text outside the kernel's domain: code point > U+024F, a capital whose lower case leaves that range, a C1 "
                                         "control, a sequence ftfy would re-decode as mojibake, or any non-ASCII byte in HF-tokenizer mode / "
                                         "the --constrain filter"),
                                     (4, "caption too long / position out of range"),
                                     (8, "sentence longer than the constraint filter accepts (511 bytes)"),
                                     (16, "constraint filter buffer overflow")) if st & bit]
            raise LeafError("tokenizer kernel: " + "; ".join(what))

    def set_deterministic(self, on: bool):
        """Bit-reproducible gradients (leaf_set_deterministic): backward() and the gradient-norm reduction sum in a fixed order
        instead of with atomics. backward() and FareTrainer follow torch.use_deterministic_algorithms on their own, so a caller
        never needs this; the forward is deterministic either way."""
        on = bool(on)
        if on != self.deterministic:
            with torch.cuda.device(self.device):
                check(self._lib.leaf_set_deterministic(self._h, 1 if on else 0))
            self.deterministic = on

    def set_tokenizer_mode(self, hf: bool):
        """hf=True: token ids of transformers' CLIPTokenizer (the reference's HF evaluation path, utils_attacks.py:67-71)
        instead of open_clip's SimpleTokenizer: no html.unescape, <|startoftext|> / <|endoftext|> spellings."""
        check(self._lib.leaf_set_tokenizer_mode(self._h, 1 if hf else 0))
        self.hf_tokenizer = bool(hf)

    def tokenize_hf(self, texts, pad_id: int = 49407) -> torch.Tensor:
        """tokenizer_wrapper.__call__ (utils_attacks.py:67-71): CLIPTokenizer(x, padding=True, truncation=True).input_ids -
        int64 [N, longest row], padded with the tokenizer's pad id after the EOS. Needs set_tokenizer_mode(True)."""
        if not getattr(self, "hf_tokenizer", False):
            raise LeafError("tokenize_hf needs set_tokenizer_mode(True)")
        if isinstance(texts, str):
            texts = [texts]
        d, o = self.upload_captions(texts)
        tok, ln, _ = self.expand_tokenize(d, o, len(texts), 0)
        self.check_status()
        # row length = index of the LAST end-of-text + 1 (a literal <|endoftext|> inside the caption is an earlier one)
        idx = torch.arange(CONTEXT_LENGTH, device=tok.device).view(1, -1)
        n_tok = torch.where(tok == 49407, idx + 1, torch.zeros_like(idx)).max(dim=1).values
        L = int(n_tok.max().item())
        tok = tok[:, :L].long()
        return torch.where(idx[:, :L] < n_tok.view(-1, 1), tok, torch.full_like(tok, pad_id))

    def encode_hf_tokens(self, tok: torch.Tensor, eos_token_id: int = 49407, normalize: bool = False) -> torch.Tensor:
        """HF CLIPTextModel(WithProjection) forward + pooling on HF-shaped rows [N, L <= 77] with any pad id: pooled at the
        FIRST eos_token_id (modeling_clip.py's rule for eos_token_id != 2; for the legacy eos_token_id == 2 configs it is
        argmax(ids), which is the same position for CLIP's vocabulary). Positions after the EOS are dead under the causal
        mask, so the pad id never matters."""
        tok = tok.to(self.device)
        N, L = tok.shape
        if L > CONTEXT_LENGTH:
            raise LeafError(f"rows longer than the context length ({L} > {CONTEXT_LENGTH})")
        is_eos = tok == eos_token_id
        if not bool(is_eos.any(dim=1).all()):
            raise LeafError("every row needs an EOS token")
        ln = (is_eos.int().argmax(dim=1) + 1).to(torch.int32)
        rows = torch.zeros((N, CONTEXT_LENGTH), dtype=torch.int32, device=self.device)
        keep = torch.arange(L, device=self.device).view(1, L) < ln.view(-1, 1)
        rows[:, :L] = torch.where(keep, tok.to(torch.int32), torch.zeros_like(tok, dtype=torch.int32))
        return self.encode_tokens(rows, ln, normalize)

    def tokenize(self, texts, check=True, with_lengths=False):
        """SimpleTokenizer.__call__ (tokenizer.py:226-265): int64 [N,77] on the engine's device. with_lengths: also the pooled
        lengths argmax(ids) + 1 as a host list - they ride on the status read, so knowing them costs no extra synchronisation
        (forward_train takes them as hints and then does not synchronise either)."""
        if isinstance(texts, str):
            texts = [texts]
        d, o = self.upload_captions(texts)
        tok, ln, _ = self.expand_tokenize(d, o, len(texts), 0)
        if with_lengths:
            both = torch.cat([self._status, ln]).cpu().tolist()              # ONE device -> host read: status flags + lengths
            if both[0]:
                self.check_status()
            return tok.long(), both[1:]
        if check:
            self.check_status()
        return tok.long()

    # ---- K2 ----------------------------------------------------------------------------------------------
    def encode_tokens(self, tok: torch.Tensor, lengths: torch.Tensor = None, normalize: bool = False,
                      base: torch.Tensor = None, dedup=(0, 0), trim: bool = False) -> torch.Tensor:
        """CLIP.encode_text (model.py:269-284) for token rows already on the device. `base` (int32 [N], -1 = none)
        names for each row another row of the batch it shares a token prefix with (computed once, results identical).
        dedup = (rows, group): the first `rows` rows come in groups of `group` candidates of one sample; duplicates
        inside a group are encoded once. trim=True: the rows after them that serve as `base` (the unedited captions) are
        computed only as far as a candidate reads them; THEIR rows of the result are undefined, all others unchanged."""
        if tok.dtype != torch.int32:
            tok = tok.to(torch.int32)
        tok = tok.contiguous()
        N = tok.shape[0]
        if lengths is None:
            lengths = (tok.argmax(dim=-1) + 1).to(torch.int32)      # transformer.py:661
        self.reserve(N)
        out = torch.empty((N, self.embed_dim), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(self._lib.leaf_encode(self._h, _ptr(tok), _ptr(lengths.contiguous()), _ptr(base), N, int(dedup[0]), int(dedup[1]), 1 if trim else 0,
                                        1 if normalize else 0, _ptr(out), _stream()))
        return out

    # ---- K4 ----------------------------------------------------------------------------------------------
    def forward_train(self, tok: torch.Tensor, lengths: torch.Tensor = None, host_lengths=None) -> torch.Tensor:
        """encode_text in train mode (utils_AT.py:317-319): same features, every layer's activations are kept. host_lengths: the
        rows' pooled lengths as a host list (tokenize(..., with_lengths=True)) - with them the call does not synchronise."""
        tok = tok.to(torch.int32).contiguous()
        N = tok.shape[0]
        if lengths is None:
            lengths = (tok.argmax(dim=-1) + 1).to(torch.int32)
        out = torch.empty((N, self.embed_dim), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(self._lib.leaf_train_reserve(self._h, N))
            gen = ctypes.c_int64(0)
            rows, longest = (sum(host_lengths), max(host_lengths)) if host_lengths is not None and len(host_lengths) == N else (0, 0)
            check(self._lib.leaf_forward_train(self._h, _ptr(tok), _ptr(lengths.contiguous()), N, _ptr(out), int(rows), int(longest),
                                               ctypes.byref(gen), _stream()))
        self.last_generation = int(gen.value)
        return out

    def backward(self, dfeat: torch.Tensor, grads: dict, generation: int = 0):
        """loss.backward() through the saved forward: ACCUMULATES into the fp32 tensors of `grads`, a dict in the same
        naming as the bound parameters (open_clip or HF); entries that are None mark frozen parameters. `generation`
        (forward_train's self.last_generation) makes the engine refuse to differentiate a forward it no longer holds."""
        if dfeat.dim() != 2 or dfeat.shape[1] != self.embed_dim:
            raise LeafError(f"dfeat must be [N, {self.embed_dim}], got {tuple(dfeat.shape)}")
        g = _canon_state(grads)
        for t in g.tensors():
            if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
                raise LeafError("gradient buffers must be contiguous fp32 CUDA tensors")
        keep = self._make_ptrs(g)
        with torch.cuda.device(self.device):
            self.set_deterministic(torch.are_deterministic_algorithms_enabled())
            check(self._lib.leaf_backward(self._h, int(generation), _ptr(dfeat.to(torch.float32).contiguous()), int(dfeat.shape[0]),
                                          ctypes.byref(keep[1]), _stream()))

    def set_backward_hook(self, fn):
        """fn(layer, user) runs on the host once backward() has enqueued a layer's gradients, and with layer -1 after the
        rest (leaf_set_backward_hook). The engine keeps the ctypes thunk alive for as long as it may call it."""
        self._backward_hook = BACKWARD_HOOK(fn)
        check(self._lib.leaf_set_backward_hook(self._h, ctypes.cast(self._backward_hook, ctypes.c_void_p), None))

    @contextlib.contextmanager
    def sm_budget(self, n_sms: int):
        """The persistent GEMM grids take at most n_sms SMs inside the block (leaf_set_sm_budget), all of them again after it."""
        check(self._lib.leaf_set_sm_budget(self._h, n_sms))
        try:
            yield
        finally:
            check(self._lib.leaf_set_sm_budget(self._h, 0))

    def adamw(self, params, grads, exp_avg, exp_avg_sq, *, n_nodecay, lr, beta1, beta2, eps, weight_decay, step, grad_scale=1.0):
        """One AdamW step (leaf_adamw) over flat fp32 buffers: grads are scaled by grad_scale, [0, n_nodecay) takes no weight decay."""
        with torch.cuda.device(self.device):
            check(self._lib.leaf_adamw(self._h, _ptr(params), _ptr(grads), _ptr(exp_avg), _ptr(exp_avg_sq), grads.numel(), n_nodecay,
                                       lr, beta1, beta2, eps, weight_decay, step, grad_scale, _stream()))

    def sumsq(self, g, out):
        """Adds the sum of squares of the flat fp32 buffer g into out[0] (leaf_sumsq; fixed-order in deterministic mode)."""
        with torch.cuda.device(self.device):
            check(self._lib.leaf_sumsq(self._h, _ptr(g), g.numel(), _ptr(out), _stream()))

    def scale(self, g, s: float):
        """g *= s in place, for a flat fp32 buffer (leaf_scale)."""
        with torch.cuda.device(self.device):
            check(self._lib.leaf_scale(self._h, _ptr(g), g.numel(), s, _stream()))

    # ---- K3 ----------------------------------------------------------------------------------------------
    def score(self, feats: torch.Tensor, anchor: torch.Tensor, B: int, n: int, objective: str = "l2", want_loss=False):
        """utils_attacks.py:332-348: returns (best int32 [B], best_feat [B,E], loss [B,n] or None)."""
        best = torch.empty((B,), dtype=torch.int32, device=self.device)
        best_feat = torch.empty((B, self.embed_dim), dtype=torch.float32, device=self.device)
        loss = torch.empty((B, n), dtype=torch.float32, device=self.device) if want_loss else None
        with torch.cuda.device(self.device):
            check(self._lib.leaf_score(self._h, _ptr(feats), _ptr(anchor), B, n, OBJECTIVES[objective], _ptr(loss), _ptr(best),
                                       _ptr(best_feat), _stream()))
        return best, best_feat, loss

    TOPK_MAX = 200 * 1024 // 4         # scores one leaf_topk launch holds in shared memory

    def topk(self, score_a: torch.Tensor, k: int, m: int = None, score_b: torch.Tensor = None):
        """Indices (int32 [k]) and values of the k largest of the first m scores; value descending, ties by ascending
        index. score_b: a second tower's scores of the same candidates, averaged in (utils_attacks.py:498-513). Longer lists
        (brute force over a caption of more than ~266 characters: (2 len + 1) * |V| candidates) go through leaf_topk in chunks
        and one more launch over the chunks' winners - equal values keep their index order through both levels."""
        score_a = score_a.reshape(-1)
        m = score_a.numel() if m is None else int(m)
        if score_b is not None:
            score_b = score_b.reshape(-1)
        if m > self.TOPK_MAX:
            idxs, vals = [], []
            for lo in range(0, m, self.TOPK_MAX):
                hi = min(m, lo + self.TOPK_MAX)
                i, v = self.topk(score_a[lo:hi], min(k, hi - lo), score_b=None if score_b is None else score_b[lo:hi])
                idxs.append(i + lo)
                vals.append(v)
            idx_all, val_all = torch.cat(idxs), torch.cat(vals).contiguous()
            if val_all.numel() > self.TOPK_MAX:
                raise LeafError(f"top-{k} of {m} scores needs more than two levels")
            pick, val = self.topk(val_all, k)
            return idx_all[pick.long()].contiguous(), val
        idx = torch.empty((k,), dtype=torch.int32, device=self.device)
        val = torch.empty((k,), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(self._lib.leaf_topk(self._h, _ptr(score_a.contiguous()), _ptr(None if score_b is None else score_b.contiguous()), m, int(k),
                                      _ptr(idx), _ptr(val), _stream()))
        return idx, val

    # ---- hooks for tests / bench ---------------------------------------------------------------------------
    def gemm(self, A, Bt, bias=None, epilogue=0, act=0, C=None, m_dev=None):
        M, K = A.shape
        N = Bt.shape[0]
        if C is None:
            C = torch.empty((M, N), dtype=torch.bfloat16 if epilogue in (0, 1) else torch.float32, device=A.device)
        with torch.cuda.device(self.device):
            check(self._lib.leaf_gemm_bf16(self._h, _ptr(A), _ptr(Bt), _ptr(bias), _ptr(C), M, N, K, epilogue, act, _ptr(m_dev), _stream()))
        return C

    def gemm_mn(self, A, B, bias=None, epilogue=3, C=None, a_mn=True):
        """B [K,N] MN-major; a_mn: A is [K,M] and C = A^T . B (the weight-gradient shape), else A is [M,K] and C = A . B
        (the data-gradient shape)."""
        K, N = B.shape
        M = A.shape[1] if a_mn else A.shape[0]
        if C is None:
            C = torch.zeros((M, N), dtype=torch.bfloat16 if epilogue in (0, 1) else torch.float32, device=A.device)
        with torch.cuda.device(self.device):
            check(self._lib.leaf_gemm_bf16_mn(self._h, _ptr(A), _ptr(B), _ptr(bias), _ptr(C), M, N, K, epilogue, 1 if a_mn else 0,
                                              _stream()))
        return C

    def test_layernorm(self, x, gamma, beta):
        y = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
        check(self._lib.leaf_test_layernorm(self._h, _ptr(x), x.shape[0], _ptr(gamma), _ptr(beta), _ptr(y), _stream()))
        return y

    def test_attention(self, qkv, meta, out=None):
        """meta int32 [N,4] = {own_row, t, p, base_row} per sequence."""
        if out is None:
            out = torch.zeros((qkv.shape[0], self.width), dtype=torch.bfloat16, device=qkv.device)
        check(self._lib.leaf_test_attention(self._h, _ptr(qkv), _ptr(meta), meta.shape[0], _ptr(out), _stream()))
        return out

    def test_attention_bwd(self, qkv, o, dout, meta, T):
        """K4's attention backward alone: dqkv bf16 [rows, 3W] = (dQ | dK | dV); meta as test_attention with p = 0."""
        dqkv = torch.zeros_like(qkv)
        check(self._lib.leaf_test_attention_bwd(self._h, _ptr(qkv), _ptr(o), _ptr(dout), _ptr(meta), meta.shape[0], int(T),
                                                _ptr(dqkv), _stream()))
        return dqkv

    def set_prune_last(self, on: bool):
        """Final-layer pruning (out-proj / MLP on the pooled EOS rows only); on by default, bit-identical either way."""
        check(self._lib.leaf_set_prune_last(self._h, 1 if on else 0))

    def launch_count(self, reset=False) -> int:
        return int(self._lib.leaf_launch_count(self._h, 1 if reset else 0))

    def set_timing(self, on: bool):
        check(self._lib.leaf_set_timing(self._h, 1 if on else 0))

    def gemm_time_ms(self):
        return self.class_time_ms(0)

    def class_time_ms(self, which: int):
        """(ms, launches) of kernel class `which` (0 GEMM, 1 LayerNorm, 2 attention, 3 packing + embedding) since
        set_timing(True): CUDA events on the launching stream around every launch of the class."""
        n = ctypes.c_int32(0)
        ms = self._lib.leaf_timing_ms(self._h, int(which), ctypes.byref(n))
        return float(ms), int(n.value)

    def last_rows(self) -> int:
        """Packed token rows (sum of argmax(ids)+1) of the last encode; synchronises."""
        return int(self._lib.leaf_last_rows(self._h))


# ---- binding a live torch module (the reference's `model` argument) ----------------------------------------------------
def _text_config(module):
    """(heads, quick_gelu, ln_eps) of an HF CLIPTextModel / CLIPTextModelWithProjection / CLIPModel from its config, or
    None when `module` is not an HF model."""
    cfg = getattr(module, "config", None)
    cfg = getattr(cfg, "text_config", None) or cfg
    act = getattr(cfg, "hidden_act", None)
    if cfg is None or act is None or not hasattr(cfg, "num_attention_heads"):
        return None
    if act not in ("quick_gelu", "gelu"):
        raise LeafError(f"unsupported text-tower activation {act!r} (the engine has nn.GELU and QuickGELU)")
    return int(cfg.num_attention_heads), act == "quick_gelu", float(getattr(cfg, "layer_norm_eps", 1e-5))


def _open_clip_config(module):
    """(heads, quick_gelu, ln_eps) of an open_clip CLIP / CustomTextCLIP / TextTransformer-shaped module: heads from the first
    residual block's nn.MultiheadAttention, the activation from the class of the MLP's activation module
    (transformer.py:33-36 QuickGELU vs nn.GELU; model.py:192)."""
    text = getattr(module, "text", module)
    blocks = getattr(getattr(text, "transformer", None), "resblocks", None)
    if blocks is None or len(blocks) == 0:
        raise LeafError("cannot find transformer.resblocks in the module (open_clip naming expected)")
    blk = blocks[0]
    heads = getattr(getattr(blk, "attn", None), "num_heads", None)
    if heads is None:
        raise LeafError("cannot infer the number of attention heads of the tower")
    acts = {type(m).__name__ for m in blk.modules()}
    quick = bool(acts & {"QuickGELU", "QuickGELUActivation"})
    if not quick and not acts & {"GELU", "GELUActivation"}:
        raise LeafError(f"cannot tell the MLP activation of the tower (module classes: {sorted(acts)})")
    eps = float(getattr(getattr(blk, "ln_1", None), "eps", 1e-5))
    return int(heads), quick, eps


def bind_module(model) -> LeafEngine:
    """Engine for a live torch module in open_clip or HF naming (also behind a DDP-style `.module` holder). Created on first
    use and cached on the module as `leaf_engine`; later calls re-cast the engine's bf16 operand copies when any bound
    parameter changed in place (optimizer step) and rebind when the parameters moved. HF layouts switch the tokenizer
    kernel to CLIPTokenizer's rules (the reference drives HF models with tokenizer_wrapper, utils_attacks.py:67-71,
    eval_textfare.py:100-127)."""
    module = model.module if isinstance(getattr(model, "module", None), torch.nn.Module) else model
    eng = getattr(module, "leaf_engine", None)
    if isinstance(eng, LeafEngine) and getattr(module, "_leaf_self_managed", False):
        return eng                                                           # LeafTextTower refreshes its own engine
    live = module.state_dict(keep_vars=True)
    v = _canon_state({k: t for k, t in live.items() if torch.is_tensor(t)})
    flat = v.tensors()
    ptrs = tuple(t.data_ptr() for t in flat)
    version = sum(t._version for t in flat)
    if isinstance(eng, LeafEngine) and getattr(eng, "_bound_ptrs", None) == ptrs:
        if eng._bound_version != version:
            eng.refresh_weights()
            eng._bound_version = version
        return eng
    heads, quick, eps = _text_config(module) or _open_clip_config(module)
    eng = LeafEngine({k: v.detach() for k, v in live.items() if torch.is_tensor(v)}, heads=heads, quick_gelu=quick, ln_eps=eps)
    if v.layout == "hf":
        eng.set_tokenizer_mode(True)
    eng._bound_ptrs, eng._bound_version = ptrs, version
    object.__setattr__(module, "leaf_engine", eng)                           # a plain attribute, not a registered submodule
    return eng

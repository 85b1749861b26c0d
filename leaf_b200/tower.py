"""LeafTextTower: a CLIP text tower whose parameters live in torch (open_clip CLIP naming, SURVEY.md appendix C)
and whose forward runs on the native engine. It offers the two duck-typed members the reference's attack uses:

    tower.encode_text(tokens, normalize=False) -> Tensor[N,E]     /root/reference/src/open_clip/model.py:269-284
    tower.tokenizer(list[str]) -> LongTensor[N,77]                 /root/reference/src/open_clip/tokenizer.py:226-265

Memory layout: every parameter is a view into ONE flat fp32 buffer, and (once trainable) every .grad a view into a
second one. The parameters the reference's optimizer puts in its weight_decay = 0 group come first
(train_AT_text_only.py:329: `p.ndim < 2 or "bn" in n or "ln" in n or "bias" in n or "logit_scale" in n`), so the FARE
update is one AdamW launch over the flat buffers, the data-parallel gradient exchange one all-reduce, and zeroing the
gradients one memset (leaf_b200/fare.py).
"""
from __future__ import annotations

import re

import torch

from . import synth
from .engine import LeafEngine


def no_weight_decay(name: str, ndim: int) -> bool:
    """train_AT_text_only.py:329."""
    return ndim < 2 or "bn" in name or "ln" in name or "bias" in name or "logit_scale" in name


class _EncodeTextTrain(torch.autograd.Function):
    """encode_text under autograd: forward = leaf_forward_train, backward = leaf_backward, which ACCUMULATES straight into
    the parameters' .grad (views of the tower's flat gradient buffer) - no per-parameter temporaries, no 390 tiny
    add kernels. The engine keeps ONE saved forward: a second encode_text with gradients enabled before this output's
    backward makes that backward raise LeafError (generation check) instead of differentiating the wrong activations. The parameters are inputs of the Function only so that autograd knows the output needs a backward."""

    @staticmethod
    def forward(ctx, tower, tok, *params):
        ctx.tower = tower
        hint, tower._host_lengths = tower._host_lengths, None                 # one-shot: set by encode_text(..., host_lengths=)
        out = tower.leaf_engine.forward_train(tok, host_lengths=hint)
        ctx.generation = tower.leaf_engine.last_generation
        return out

    @staticmethod
    def backward(ctx, dfeat):
        tower = ctx.tower
        tower.attach_grads()
        grads = {k: (p.grad if p.requires_grad else None) for k, p in tower.named_tower_parameters()}
        tower.leaf_engine.backward(dfeat, grads, ctx.generation)
        return (None, None) + (None,) * len(grads)


_TEXT_KEYS = re.compile(r"^(?:module\.)?(?:text\.)?(?P<key>token_embedding\.weight|positional_embedding|ln_final\.(weight|bias)|"
                        r"text_projection(\.weight)?|"
                        r"transformer\.resblocks\.\d+\.(ln_1|ln_2|attn\.out_proj|mlp\.c_fc|mlp\.c_proj)\.(weight|bias)|"
                        r"transformer\.resblocks\.\d+\.attn\.in_proj_(weight|bias))$")


def text_tower_state_dict(state_dict: dict) -> dict:
    """The text-tower entries of an open_clip CLIP / CustomTextCLIP state dict (SURVEY.md appendix C): everything under
    `visual.`, `logit_scale`, the attention-mask buffer etc. is dropped; a `text.` prefix, and the `module.` prefix of a
    state dict saved through DDP, are removed."""
    out = {}
    for k, v in state_dict.items():
        m = _TEXT_KEYS.match(k)
        if m:
            out[m["key"]] = v
    return out


def open_clip_to_hf(sd: dict) -> dict:
    """The reference's export mapping (conversion/convert_2.py:37-99, copy_text_model_and_projection): an open_clip text-tower
    state dict -> the keys of transformers' CLIPTextModelWithProjection (equally the text half of a CLIPModel): fused
    in_proj split into q / k / v (`chunk(3, dim=0)`, :39-40), c_fc / c_proj -> fc1 / fc2, ln_1 / ln_2 -> layer_norm1 / 2,
    positional_embedding -> position_embedding.weight, text_projection [W,E] -> text_projection.weight = P^T [E,W] (:85).
    Tensors are new (contiguous copies), on the source's device."""
    sd = text_tower_state_dict(sd)
    out = {"text_model.embeddings.token_embedding.weight": sd["token_embedding.weight"].clone(),
           "text_model.embeddings.position_embedding.weight": sd["positional_embedding"].clone(),
           "text_model.final_layer_norm.weight": sd["ln_final.weight"].clone(),
           "text_model.final_layer_norm.bias": sd["ln_final.bias"].clone(),
           "text_projection.weight": sd["text_projection"].t().contiguous()}
    i = 0
    while f"transformer.resblocks.{i}.ln_1.weight" in sd:
        p, q = f"transformer.resblocks.{i}.", f"text_model.encoder.layers.{i}."
        for nm, w, b in zip("qkv", sd[p + "attn.in_proj_weight"].chunk(3, dim=0), sd[p + "attn.in_proj_bias"].chunk(3, dim=0)):
            out[q + f"self_attn.{nm}_proj.weight"], out[q + f"self_attn.{nm}_proj.bias"] = w.contiguous().clone(), b.contiguous().clone()
        for a, b in (("attn.out_proj", "self_attn.out_proj"), ("ln_1", "layer_norm1"), ("ln_2", "layer_norm2"),
                     ("mlp.c_fc", "mlp.fc1"), ("mlp.c_proj", "mlp.fc2")):
            out[q + b + ".weight"], out[q + b + ".bias"] = sd[p + a + ".weight"].clone(), sd[p + a + ".bias"].clone()
        i += 1
    return out


def hf_to_open_clip(sd: dict) -> dict:
    """The inverse mapping (the direction of the reference's convert_to_openclip.py): HF CLIPTextModel(WithProjection) /
    CLIPModel keys -> an open_clip text-tower state dict LeafTextTower accepts."""
    pre = next((k[: -len("embeddings.token_embedding.weight")] for k in sd if k.endswith("embeddings.token_embedding.weight")), None)
    if pre is None:
        raise ValueError("not an HF CLIP text state dict (no embeddings.token_embedding.weight)")
    root = pre[: -len("text_model.")] if pre.endswith("text_model.") else pre
    out = {"token_embedding.weight": sd[pre + "embeddings.token_embedding.weight"].clone(),
           "positional_embedding": sd[pre + "embeddings.position_embedding.weight"].clone(),
           "ln_final.weight": sd[pre + "final_layer_norm.weight"].clone(), "ln_final.bias": sd[pre + "final_layer_norm.bias"].clone(),
           "text_projection": sd[root + "text_projection.weight"].t().contiguous()}
    i = 0
    while (pre + f"encoder.layers.{i}.layer_norm1.weight") in sd:
        q, p = pre + f"encoder.layers.{i}.", f"transformer.resblocks.{i}."
        out[p + "attn.in_proj_weight"] = torch.cat([sd[q + f"self_attn.{nm}_proj.weight"] for nm in "qkv"], dim=0)
        out[p + "attn.in_proj_bias"] = torch.cat([sd[q + f"self_attn.{nm}_proj.bias"] for nm in "qkv"], dim=0)
        for a, b in (("attn.out_proj", "self_attn.out_proj"), ("ln_1", "layer_norm1"), ("ln_2", "layer_norm2"),
                     ("mlp.c_fc", "mlp.fc1"), ("mlp.c_proj", "mlp.fc2")):
            out[p + a + ".weight"], out[p + a + ".bias"] = sd[q + b + ".weight"].clone(), sd[q + b + ".bias"].clone()
        i += 1
    return out


class LeafTextTower(torch.nn.Module):
    _leaf_self_managed = True            # engine.bind_module: this module refreshes its own engine (refresh())

    def __init__(self, state_dict: dict, heads: int, quick_gelu: bool = False, device="cuda"):
        super().__init__()
        state_dict = text_tower_state_dict(state_dict)
        if "token_embedding.weight" not in state_dict:
            raise ValueError("LeafTextTower needs an open_clip text tower state dict (token_embedding.weight, ...)")
        items = sorted(state_dict.items(), key=lambda kv: 0 if no_weight_decay(kv[0], kv[1].dim()) else 1)   # stable
        sizes = [(v.numel() + 3) // 4 * 4 for _, v in items]                     # 16-byte aligned slices
        self._flat = torch.zeros(sum(sizes), dtype=torch.float32, device=device)
        self._gflat = None
        self._names, self._slices = {}, {}
        off = 0
        self.n_nodecay = 0
        for (k, v), sz in zip(items, sizes):
            view = self._flat[off:off + v.numel()].view(v.shape)
            view.copy_(v.detach().to(device=device, dtype=torch.float32))
            safe = k.replace(".", "__")
            self._names[k] = safe
            self._slices[k] = (off, v.numel(), tuple(v.shape))
            self.register_parameter(safe, torch.nn.Parameter(view, requires_grad=False))
            off += sz
            if no_weight_decay(k, v.dim()):
                self.n_nodecay = off
        self.heads, self.quick_gelu = heads, quick_gelu
        self._host_lengths = None
        self.leaf_engine = LeafEngine(self.open_clip_state_dict(), heads=heads, quick_gelu=quick_gelu)

    @classmethod
    def random(cls, name_or_cfg, seed: int = 0, device="cuda", exact_numpy: bool = False):
        """Random-init tower of a named shape (synth.TOWERS; init rule of transformer.py:731-752)."""
        cfg = synth.TOWERS[name_or_cfg] if isinstance(name_or_cfg, str) else name_or_cfg
        sd = synth.random_tower_state_dict(cfg, seed=seed, device="cpu" if exact_numpy else device, exact_numpy=exact_numpy)
        return cls(sd, heads=cfg.heads, quick_gelu=cfg.quick_gelu, device=device)

    @classmethod
    def from_hf(cls, hf_model, device="cuda"):
        """A trainable LeafTextTower from a transformers CLIPTextModelWithProjection / CLIPModel (weights COPIED into the flat
        buffer; export back with hf_state_dict / load_into_hf)."""
        cfg = getattr(hf_model.config, "text_config", None) or hf_model.config
        if cfg.hidden_act not in ("gelu", "quick_gelu"):
            raise ValueError(f"unsupported activation {cfg.hidden_act!r}")
        sd = hf_to_open_clip({k: v.detach() for k, v in hf_model.state_dict().items()})
        return cls(sd, heads=int(cfg.num_attention_heads), quick_gelu=cfg.hidden_act == "quick_gelu", device=device)

    def hf_state_dict(self) -> dict:
        """The tower's CURRENT parameters under transformers' CLIPTextModelWithProjection keys - the reference's HF
        checkpoint export (conversion/convert_2.py:37-99) for a tower trained here."""
        return open_clip_to_hf(self.open_clip_state_dict())

    def hf_text_config(self, **overrides):
        """transformers.CLIPTextConfig of this tower (what conversion/convert_2.py builds from the open_clip config)."""
        from transformers import CLIPTextConfig
        e = self.leaf_engine
        kw = dict(vocab_size=int(self._slices["token_embedding.weight"][2][0]), hidden_size=e.width, intermediate_size=4 * e.width,
                  num_hidden_layers=e.layers, num_attention_heads=e.heads, max_position_embeddings=int(self._slices["positional_embedding"][2][0]),
                  hidden_act="quick_gelu" if self.quick_gelu else "gelu", projection_dim=e.embed_dim, layer_norm_eps=1e-5,
                  bos_token_id=49406, eos_token_id=49407, pad_token_id=49407)
        kw.update(overrides)
        return CLIPTextConfig(**kw)

    def load_into_hf(self, hf_model=None):
        """Copy the parameters into `hf_model` (a CLIPTextModelWithProjection, or the text half of a CLIPModel:
        strict=False leaves its vision tower alone); with None a fresh CLIPTextModelWithProjection is built."""
        if hf_model is None:
            from transformers import CLIPTextModelWithProjection
            hf_model = CLIPTextModelWithProjection(self.hf_text_config())
        missing, unexpected = hf_model.load_state_dict(self.hf_state_dict(), strict=False)
        if unexpected or any("text_model" in k or k.startswith("text_projection") for k in missing):
            raise ValueError(f"HF export does not fit the target model: missing {missing}, unexpected {unexpected}")
        return hf_model

    # ---- parameters ------------------------------------------------------------------------------------------
    def named_tower_parameters(self):
        return [(k, getattr(self, safe)) for k, safe in self._names.items()]

    def open_clip_state_dict(self) -> dict:
        return {k: getattr(self, safe).data for k, safe in self._names.items()}

    def load_open_clip_state_dict(self, state_dict: dict):
        """The inverse of open_clip_state_dict(): copies the text-tower entries of `state_dict` (any key form
        text_tower_state_dict accepts: a whole CLIP state dict, a `text.` or a DDP `module.` prefix) IN PLACE into the flat
        buffer, so the .grad views and a FareTrainer's references stay valid, then re-casts the engine's operand copies.
        Names and shapes are checked before anything is copied: ValueError lists the missing, unexpected and mis-shaped keys."""
        sd = text_tower_state_dict(state_dict)
        bad = [f"missing: {k}" for k in self._slices if k not in sd]
        bad += [f"unexpected: {k}" for k in sd if k not in self._slices]
        bad += [f"shape of {k}: {tuple(v.shape)}, this tower has {self._slices[k][2]}" for k, v in sd.items()
                if k in self._slices and tuple(v.shape) != self._slices[k][2]]
        if bad:
            raise ValueError("state dict does not fit this LeafTextTower: " + "; ".join(bad))
        with torch.no_grad():
            for k, (off, n, shape) in self._slices.items():
                self._flat[off:off + n].view(shape).copy_(sd[k])
        self.refresh()

    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):
        """nn.Module.load_state_dict (this module's own parameter names), followed by refresh(): without it the engine would
        keep computing with its operand copies of the old weights. assign=True would replace the parameters, which are
        views of the flat buffer the engine and the optimizer read, and is refused."""
        if assign:
            raise ValueError("LeafTextTower parameters are views of one flat buffer: load_state_dict(assign=True) would detach them")
        try:
            return super().load_state_dict(state_dict, strict=strict)
        finally:                                  # torch copies every entry that fits before it raises on the others
            self.refresh()

    @property
    def flat_params(self) -> torch.Tensor:
        return self._flat

    @property
    def flat_grads(self) -> torch.Tensor:
        if self._gflat is None:
            self._gflat = torch.zeros_like(self._flat)
        return self._gflat

    def attach_grads(self):
        """Make every trainable parameter's .grad the matching view of the flat gradient buffer. A .grad that is None
        (fresh, or after optimizer.zero_grad(set_to_none=True)) starts from zero."""
        g = self.flat_grads
        params = [(k, p) for k, p in self.named_tower_parameters() if p.requires_grad]
        if all(p.grad is None for _, p in params):
            g.zero_()
        for k, p in params:
            off, n, shape = self._slices[k]
            view = g[off:off + n].view(shape)
            if p.grad is None:
                if not all(q.grad is None for _, q in params):
                    view.zero_()
                p.grad = view
            elif p.grad.data_ptr() != view.data_ptr():
                view.copy_(p.grad)
                p.grad = view

    def zero_grad(self, set_to_none: bool = False):
        """One memset of the flat buffer; the .grad views stay attached."""
        if self._gflat is not None:
            self._gflat.zero_()
        if set_to_none:
            for p in self.parameters():
                p.grad = None

    def refresh(self):
        """Call after the parameters changed (optimizer step)."""
        self.leaf_engine.refresh_weights()

    def tokenizer(self, texts, with_lengths=False):
        return self.leaf_engine.tokenize(texts, with_lengths=with_lengths)

    def trainable(self, on: bool = True):
        """Mark the tower's parameters as requiring gradients (the attacked tower in train_AT_text_only.py)."""
        for p in self.parameters():
            p.requires_grad_(on)
        return self

    def encode_text(self, text, normalize: bool = False, host_lengths=None):
        """model.py:269-284. host_lengths (training path only): the rows' pooled lengths as a host list, from
        tokenizer(texts, with_lengths=True) - the train-mode forward then needs no stream synchronisation. Under torch.no_grad() (the attack, utils_AT.py:295) this is the inference path; with
        gradients enabled and trainable parameters (utils_AT.py:317-319) the forward keeps its activations and
        loss.backward() runs the engine's backward. Call refresh() after optimizer.step()."""
        params = [p for _, p in self.named_tower_parameters()]
        if torch.is_grad_enabled() and any(p.requires_grad for p in params):
            self._host_lengths = host_lengths
            f = _EncodeTextTrain.apply(self, text, *params)
            return torch.nn.functional.normalize(f, dim=-1) if normalize else f
        with torch.no_grad():
            return self.leaf_engine.encode_tokens(text, None, normalize)

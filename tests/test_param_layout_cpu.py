"""The tower's parameter names (leaf_b200/_native.py: TOWER_PARAMS, LAYER_PARAMS) and what is built from them, on CPU tensors:
engine._canon_state binds every ABI field to the tensor of the key spelled out below in each naming the engine accepts,
text_tower_state_dict keeps the tower's entries in input order, and the two converters invert each other with the key
order they have always written."""
import pytest
import torch

from leaf_b200 import LeafError, synth
from leaf_b200.engine import _canon_state
from leaf_b200.tower import hf_to_open_clip, open_clip_to_hf, text_tower_state_dict
from tests.test_gpu_dropin import OpenClipNamedTower, _hf_text_config

OPEN_CLIP_TOP = {"token_embedding": "token_embedding.weight", "positional_embedding": "positional_embedding",
                 "lnf_w": "ln_final.weight", "lnf_b": "ln_final.bias", "text_projection": "text_projection"}
OPEN_CLIP_LAYER = {"ln1_w": "ln_1.weight", "ln1_b": "ln_1.bias", "in_proj_w": "attn.in_proj_weight", "in_proj_b": "attn.in_proj_bias",
                   "out_w": "attn.out_proj.weight", "out_b": "attn.out_proj.bias", "ln2_w": "ln_2.weight", "ln2_b": "ln_2.bias",
                   "fc1_w": "mlp.c_fc.weight", "fc1_b": "mlp.c_fc.bias", "fc2_w": "mlp.c_proj.weight", "fc2_b": "mlp.c_proj.bias"}
HF_TOP = {"token_embedding": "text_model.embeddings.token_embedding.weight",
          "positional_embedding": "text_model.embeddings.position_embedding.weight",
          "lnf_w": "text_model.final_layer_norm.weight", "lnf_b": "text_model.final_layer_norm.bias",
          "text_projection": "text_projection.weight"}
HF_LAYER = {"ln1_w": "layer_norm1.weight", "ln1_b": "layer_norm1.bias",
            "q_w": "self_attn.q_proj.weight", "k_w": "self_attn.k_proj.weight", "v_w": "self_attn.v_proj.weight",
            "q_b": "self_attn.q_proj.bias", "k_b": "self_attn.k_proj.bias", "v_b": "self_attn.v_proj.bias",
            "out_w": "self_attn.out_proj.weight", "out_b": "self_attn.out_proj.bias", "ln2_w": "layer_norm2.weight",
            "ln2_b": "layer_norm2.bias", "fc1_w": "mlp.fc1.weight", "fc1_b": "mlp.fc1.bias", "fc2_w": "mlp.fc2.weight",
            "fc2_b": "mlp.fc2.bias"}

# what open_clip_to_hf and hf_to_open_clip wrote for a two-layer tower before they were derived from the table
OPEN_CLIP_TO_HF_KEYS = [
    "text_model.embeddings.token_embedding.weight", "text_model.embeddings.position_embedding.weight",
    "text_model.final_layer_norm.weight", "text_model.final_layer_norm.bias", "text_projection.weight",
    "text_model.encoder.layers.0.self_attn.q_proj.weight", "text_model.encoder.layers.0.self_attn.q_proj.bias",
    "text_model.encoder.layers.0.self_attn.k_proj.weight", "text_model.encoder.layers.0.self_attn.k_proj.bias",
    "text_model.encoder.layers.0.self_attn.v_proj.weight", "text_model.encoder.layers.0.self_attn.v_proj.bias",
    "text_model.encoder.layers.0.self_attn.out_proj.weight", "text_model.encoder.layers.0.self_attn.out_proj.bias",
    "text_model.encoder.layers.0.layer_norm1.weight", "text_model.encoder.layers.0.layer_norm1.bias",
    "text_model.encoder.layers.0.layer_norm2.weight", "text_model.encoder.layers.0.layer_norm2.bias",
    "text_model.encoder.layers.0.mlp.fc1.weight", "text_model.encoder.layers.0.mlp.fc1.bias",
    "text_model.encoder.layers.0.mlp.fc2.weight", "text_model.encoder.layers.0.mlp.fc2.bias",
    "text_model.encoder.layers.1.self_attn.q_proj.weight", "text_model.encoder.layers.1.self_attn.q_proj.bias",
    "text_model.encoder.layers.1.self_attn.k_proj.weight", "text_model.encoder.layers.1.self_attn.k_proj.bias",
    "text_model.encoder.layers.1.self_attn.v_proj.weight", "text_model.encoder.layers.1.self_attn.v_proj.bias",
    "text_model.encoder.layers.1.self_attn.out_proj.weight", "text_model.encoder.layers.1.self_attn.out_proj.bias",
    "text_model.encoder.layers.1.layer_norm1.weight", "text_model.encoder.layers.1.layer_norm1.bias",
    "text_model.encoder.layers.1.layer_norm2.weight", "text_model.encoder.layers.1.layer_norm2.bias",
    "text_model.encoder.layers.1.mlp.fc1.weight", "text_model.encoder.layers.1.mlp.fc1.bias",
    "text_model.encoder.layers.1.mlp.fc2.weight", "text_model.encoder.layers.1.mlp.fc2.bias",
]
HF_TO_OPEN_CLIP_KEYS = [
    "token_embedding.weight", "positional_embedding", "ln_final.weight", "ln_final.bias", "text_projection",
    "transformer.resblocks.0.attn.in_proj_weight", "transformer.resblocks.0.attn.in_proj_bias",
    "transformer.resblocks.0.attn.out_proj.weight", "transformer.resblocks.0.attn.out_proj.bias",
    "transformer.resblocks.0.ln_1.weight", "transformer.resblocks.0.ln_1.bias", "transformer.resblocks.0.ln_2.weight",
    "transformer.resblocks.0.ln_2.bias", "transformer.resblocks.0.mlp.c_fc.weight", "transformer.resblocks.0.mlp.c_fc.bias",
    "transformer.resblocks.0.mlp.c_proj.weight", "transformer.resblocks.0.mlp.c_proj.bias",
    "transformer.resblocks.1.attn.in_proj_weight", "transformer.resblocks.1.attn.in_proj_bias",
    "transformer.resblocks.1.attn.out_proj.weight", "transformer.resblocks.1.attn.out_proj.bias",
    "transformer.resblocks.1.ln_1.weight", "transformer.resblocks.1.ln_1.bias", "transformer.resblocks.1.ln_2.weight",
    "transformer.resblocks.1.ln_2.bias", "transformer.resblocks.1.mlp.c_fc.weight", "transformer.resblocks.1.mlp.c_fc.bias",
    "transformer.resblocks.1.mlp.c_proj.weight", "transformer.resblocks.1.mlp.c_proj.bias",
]


def _open_clip(seed=23):
    return synth.random_tower_state_dict(synth.TOWERS["tiny"], seed=seed, exact_numpy=True)


def _linear_projection(sd):
    """The same tower with open_clip's nn.Linear projection: text_projection.weight = P^T, [E, W]."""
    out = dict(sd)
    out["text_projection.weight"] = out.pop("text_projection").t().contiguous()
    return out


def _hf_models():
    from transformers import CLIPConfig, CLIPModel, CLIPTextModel, CLIPTextModelWithProjection, CLIPVisionConfig
    torch.manual_seed(0)
    tcfg = _hf_text_config(False, layers=3, W=128, heads=2, E=64)
    vcfg = CLIPVisionConfig(hidden_size=64, intermediate_size=128, num_hidden_layers=1, num_attention_heads=2, image_size=32, patch_size=16)
    return {"with_projection": CLIPTextModelWithProjection(tcfg), "text_model": CLIPTextModel(tcfg),
            "clip_model": CLIPModel(CLIPConfig(text_config=tcfg.to_dict(), vision_config=vcfg.to_dict(), projection_dim=64))}


def _check_view(sd, top, layer, layer_prefix, n_layers, projection_is_ew, synthesised=False):
    v = _canon_state(sd)
    assert len(v.layers) == n_layers
    assert v.projection_is_ew == projection_is_ew and v.projection_synthesised == synthesised
    assert list(v.top) == list(top)
    for f, k in top.items():
        if not (synthesised and f == "text_projection"):
            assert v.top[f] is sd[k], f
    for i in (0, n_layers - 1):
        assert sorted(v.layers[i]) == sorted(layer), i
        for f, k in layer.items():
            assert v.layers[i][f] is sd[layer_prefix.format(i) + k], (i, f)
    return v


def test_open_clip_forms_bind_every_field_to_its_key():
    sd = _open_clip()
    _check_view(sd, OPEN_CLIP_TOP, OPEN_CLIP_LAYER, "transformer.resblocks.{}.", 2, 0)

    text = {"text." + k: t for k, t in sd.items()}                          # CustomTextCLIP keeps its tower under .text
    _check_view(text, {f: "text." + k for f, k in OPEN_CLIP_TOP.items()}, OPEN_CLIP_LAYER, "text.transformer.resblocks.{}.", 2, 0)

    lin = _linear_projection(sd)
    v = _check_view(lin, dict(OPEN_CLIP_TOP, text_projection="text_projection.weight"), OPEN_CLIP_LAYER,
                    "transformer.resblocks.{}.", 2, 1)
    assert v.top["text_projection"].shape == (64, 128)

    ddp = {"module." + k: t for k, t in sd.items()}
    with pytest.raises(LeafError, match="naming"):                           # the binder does not strip DDP's prefix itself
        _canon_state(ddp)
    stripped = text_tower_state_dict(ddp)                                    # LeafTextTower's route
    v = _check_view(stripped, OPEN_CLIP_TOP, OPEN_CLIP_LAYER, "transformer.resblocks.{}.", 2, 0)
    assert v.top["token_embedding"] is sd["token_embedding.weight"]


def test_hf_models_bind_every_field_to_its_key():
    for kind, m in _hf_models().items():
        sd = m.state_dict(keep_vars=True)
        v = _check_view(sd, HF_TOP, HF_LAYER, "text_model.encoder.layers.{}.", 3, 1, synthesised=kind == "text_model")
        assert v.layout == "hf"
        if kind == "text_model":                         # pooler_output: an identity head the dict does not hold
            assert torch.equal(v.top["text_projection"], torch.eye(128))
            assert all(t is not v.top["text_projection"] for t in v.tensors())
        assert len(v.tensors()) == 4 + (kind != "text_model") + 3 * 16


def test_neither_naming_is_refused():
    with pytest.raises(LeafError, match="naming"):
        _canon_state({"weight": torch.zeros(2), "visual.proj": torch.zeros(2, 2)})


def test_text_tower_state_dict_keeps_input_order_and_drops_the_rest():
    tower = OpenClipNamedTower(synth.TOWERS["tiny"])
    own = tower.state_dict()                             # positional_embedding, text_projection, logit_scale, token_embedding, ...
    junk = {"visual.conv1.weight": torch.zeros(4, 3, 2, 2), "visual.proj": torch.zeros(4, 2), "logit_scale": torch.ones([]),
            "attn_mask": torch.zeros(77, 77), "text_projection.bias": torch.zeros(64), "transformer.resblocks.0.attn.bias_k": torch.zeros(1)}
    sd = {"visual.conv1.weight": junk["visual.conv1.weight"]}
    sd.update(own)
    sd.update(junk)
    want = [k for k in sd if k not in junk]
    assert len(want) == 5 + 2 * 12 and list(own).index("logit_scale") == 2
    for prefix in ("", "text.", "module.", "module.text."):
        got = text_tower_state_dict({prefix + k: t for k, t in sd.items()})
        assert list(got) == want, prefix
        assert all(got[k] is sd[k] for k in want)
    lin = text_tower_state_dict(_linear_projection(_open_clip()))
    assert "text_projection.weight" in lin and "text_projection" not in lin


def _bits(t):
    return t.contiguous().view(torch.int32)


def test_converters_invert_each_other_and_keep_their_key_order():
    sd = _open_clip()
    hf = open_clip_to_hf(sd)
    assert list(hf) == OPEN_CLIP_TO_HF_KEYS
    back = hf_to_open_clip(hf)
    assert list(back) == HF_TO_OPEN_CLIP_KEYS
    assert sorted(back) == sorted(sd)
    for k, t in sd.items():
        assert torch.equal(_bits(back[k]), _bits(t)), k
    src = {t.data_ptr() for t in sd.values()}
    assert not any(t.data_ptr() in src for t in hf.values())                  # copies, not views of the source
    assert not any(t.data_ptr() in {u.data_ptr() for u in hf.values()} for t in back.values())

    lin = open_clip_to_hf(_linear_projection(sd))                             # nn.Linear's projection: the same export
    assert list(lin) == OPEN_CLIP_TO_HF_KEYS
    assert all(torch.equal(_bits(lin[k]), _bits(hf[k])) for k in hf)

    models = _hf_models()
    clip = hf_to_open_clip(models["clip_model"].state_dict())                 # text half of a CLIPModel; vision keys ignored
    assert list(clip)[:5] == HF_TO_OPEN_CLIP_KEYS[:5] and len(clip) == 5 + 3 * 12
    with pytest.raises(ValueError, match="projection"):                       # CLIPTextModel: nothing to export as text_projection
        hf_to_open_clip(models["text_model"].state_dict())

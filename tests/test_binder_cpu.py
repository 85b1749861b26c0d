"""The drop-in binder's model introspection (leaf_b200/engine.py: _text_config, _open_clip_config, _canon_state) on CPU modules -
no engine is created, so this runs without a GPU: the activation comes from the HF config or from the open_clip module classes
(round 1 matched the class NAME "QuickGELU" only and bound every transformers quick_gelu model as erf-GELU), heads and LayerNorm
eps likewise; layouts are recognised by their parameter names, behind a `text.` prefix too; anything else fails loudly."""
import pytest
import torch

from leaf_b200 import LeafError, synth
from leaf_b200.engine import _canon_state, _open_clip_config, _text_config
from tests.test_gpu_dropin import OpenClipNamedTower, _hf_text_config


def test_hf_config_detection():
    from transformers import CLIPConfig, CLIPModel, CLIPTextModel, CLIPTextModelWithProjection, CLIPVisionConfig
    vcfg = CLIPVisionConfig(hidden_size=64, intermediate_size=128, num_hidden_layers=1, num_attention_heads=2, image_size=32, patch_size=16)
    for quick in (False, True):
        tcfg = _hf_text_config(quick, layers=1, W=128, heads=2, E=64)
        for m in (CLIPTextModelWithProjection(tcfg), CLIPTextModel(tcfg),
                  CLIPModel(CLIPConfig(text_config=tcfg.to_dict(), vision_config=vcfg.to_dict(), projection_dim=64))):
            assert _text_config(m) == (2, quick, 1e-5), type(m).__name__
            if not isinstance(m, CLIPModel):      # (a CLIPModel's VISION tower has its own activation: scanning all modules would be wrong)
                assert any(type(x).__name__ == "QuickGELUActivation" for x in m.modules()) == quick     # the class round 1 missed
            c = _canon_state({k: v for k, v in m.state_dict(keep_vars=True).items()})
            assert c.layout == "hf" and len(c.layers) == 1 and c.top["token_embedding"].shape == (49408, 128)
            assert c.projection_synthesised == isinstance(m, CLIPTextModel)                            # pooler_output: identity head
    bad = _hf_text_config(False, layers=1, W=128, heads=2, E=64)
    bad.hidden_act = "gelu_new"
    with pytest.raises(LeafError, match="activation"):
        _text_config(CLIPTextModel(bad))
    assert _text_config(torch.nn.Linear(2, 2)) is None


def test_open_clip_module_detection():
    cfg = synth.TOWERS["tiny"]
    for quick in (False, True):
        tower = OpenClipNamedTower(cfg, quick=quick)
        assert _open_clip_config(tower) == (cfg.heads, quick, 1e-5)
        holder = torch.nn.Module()
        holder.text = tower                                                       # CustomTextCLIP keeps its tower under `.text`
        assert _open_clip_config(holder) == (cfg.heads, quick, 1e-5)
        c = _canon_state({k: v for k, v in holder.state_dict(keep_vars=True).items()})
        assert c.layout == "open_clip" and len(c.layers) == cfg.layers and c.projection_is_ew == 0
    with pytest.raises(LeafError):
        _open_clip_config(torch.nn.Linear(2, 2))
    with pytest.raises(LeafError, match="naming"):
        _canon_state({"weight": torch.zeros(2)})


def test_real_open_clip_models_are_recognised():
    """The reference's own model classes (open_clip.create_model through oracle/ref_shims) from a LIONS-EPFL/LEAF checkout named
    by LEAF_REFERENCE (not part of this repository, so skipped without it): CLIP with nn.GELU and with QuickGELU, heads, eps,
    layout, and the DDP-style holder. tests/test_gpu_dropin.py's OpenClipNamedTower stands in for these classes elsewhere."""
    import os
    import subprocess
    import sys
    ref = os.environ.get("LEAF_REFERENCE", "")
    if not ref or not os.path.isdir(os.path.join(ref, "src", "open_clip")):
        pytest.skip("set LEAF_REFERENCE to a LIONS-EPFL/LEAF checkout to run this test")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = r'''
import sys, torch
sys.path[:0] = [ROOT + "/oracle/ref_shims", REF + "/src", REF, ROOT]
import open_clip
from leaf_b200.engine import _canon_state, _open_clip_config
for name, quick, heads, layers, width in (("ViT-B-32", False, 8, 12, 512), ("ViT-B-32-quickgelu", True, 8, 12, 512), ("ViT-L-14", False, 12, 12, 768)):
    m = open_clip.create_model(name, pretrained=None)
    assert _open_clip_config(m) == (heads, quick, 1e-5), (name, _open_clip_config(m))
    holder = torch.nn.Module(); holder.module = m
    c = _canon_state({k: v for k, v in m.state_dict(keep_vars=True).items()})
    assert c.layout == "open_clip" and len(c.layers) == layers and c.top["token_embedding"].shape[1] == width and c.projection_is_ew == 0
print("OK")
'''.replace("ROOT", repr(root)).replace("REF", repr(ref))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "OK" in out.stdout, out.stderr[-3000:]

"""Drop-in surface against the reference's `llava` package (SURVEY 4(iv), llava_arch.py:29-41,141-144; llava_qwen.py:37-56).

The checkpoint key names come from the reference model (tests/golden/llava_model_keys.txt, oracle/gen_golden_llava.py).
`patch_llava()` swaps the two factories and encode_images inside an importable `llava` package; here that package is a
stand-in with the reference's module layout, so the test runs without the reference tree.  A model built through the
patched factory names must hold the B200 modules, load the fixture strictly, and dispatch encode_images to the library
(which, on a CPU-only host, fails loudly -- there is no fallback)."""
import os
import sys
import types

import pytest
import torch

import ml_fastvlm_b200 as pkg
from oracle import fixture as fx


def test_model_state_dict_keys_match_reference_model(golden_dir, tower_sd, proj_sd):
    """Runs anywhere: the key names a released checkpoint uses for the path (recorded from the reference model by
    oracle/gen_golden_llava.py) == `model.vision_tower.` + our tower keys, `model.mm_projector.` + our projector keys."""
    want = [l.strip() for l in open(os.path.join(golden_dir, "llava_model_keys.txt")) if l.strip()]

    class Args:
        mm_vision_tower = "mobileclip_l_256"
        unfreeze_mm_vision_tower = False
        mm_projector_type = "mlp2x_gelu"
        mm_hidden_size = 3072
        hidden_size = 128
    tower = pkg.build_vision_tower(Args())
    proj = pkg.build_vision_projector(Args())
    got = ["model.vision_tower." + k for k in tower.state_dict().keys()] + ["model.mm_projector." + k for k in proj.state_dict().keys()]
    assert sorted(got) == sorted(want)


def _stand_in_llava(monkeypatch):
    """The three modules of apple/ml-fastvlm's `llava` package that patch_llava() edits, as empty stand-ins whose factories
    and encode_images fail if they are still called after the patch."""
    def unpatched(*args, **kwargs):
        raise AssertionError("the original factory was called")

    class LlavaMetaForCausalLM:
        def encode_images(self, images):
            raise AssertionError("the original encode_images was called")

    names = ["llava", "llava.model", "llava.model.llava_arch", "llava.model.multimodal_encoder", "llava.model.multimodal_encoder.builder",
             "llava.model.multimodal_projector", "llava.model.multimodal_projector.builder"]
    mods = {n: types.ModuleType(n) for n in names}
    for n, m in mods.items():
        monkeypatch.setitem(sys.modules, n, m)
        if "." in n:
            parent, leaf = n.rsplit(".", 1)
            setattr(mods[parent], leaf, m)
    mods["llava.model.multimodal_encoder.builder"].build_vision_tower = unpatched
    mods["llava.model.multimodal_projector.builder"].build_vision_projector = unpatched
    mods["llava.model.llava_arch"].build_vision_tower = unpatched
    mods["llava.model.llava_arch"].build_vision_projector = unpatched
    mods["llava.model.llava_arch"].LlavaMetaForCausalLM = LlavaMetaForCausalLM
    return mods


def test_patch_llava_installs_b200_modules(monkeypatch, golden_dir, tower_sd):
    mods = _stand_in_llava(monkeypatch)
    llava_arch = pkg.patch_llava()
    assert llava_arch is mods["llava.model.llava_arch"]
    assert mods["llava.model.multimodal_encoder.builder"].build_vision_tower is pkg.build_vision_tower
    assert mods["llava.model.multimodal_projector.builder"].build_vision_projector is pkg.build_vision_projector

    class Config:
        mm_vision_tower = "mobileclip_l_256"
        mm_projector_type = "mlp2x_gelu"
        mm_hidden_size = 3072
        hidden_size = 128
        unfreeze_mm_vision_tower = True          # materialise the tower despite delay_load (mobileclip_encoder.py:23-26)

    class TinyLlava(torch.nn.Module, llava_arch.LlavaMetaForCausalLM):
        """Builds its modules through the module-level factory names, as LlavaMetaModel.__init__ does (llava_arch.py:30-36)."""

        def __init__(self, cfg):
            super().__init__()
            self.vision_tower = llava_arch.build_vision_tower(cfg, delay_load=True)
            self.mm_projector = llava_arch.build_vision_projector(cfg)

        def get_model(self):
            return self

        def get_vision_tower(self):
            return self.vision_tower

    torch.manual_seed(0)
    model = TinyLlava(Config()).eval()
    tower = model.get_model().get_vision_tower()
    proj = model.get_model().mm_projector
    assert isinstance(tower, pkg.FastViTHDVisionTower) and isinstance(proj, pkg.FastVLMProjector)
    # the fixture under the reference model's key names loads strictly (the stand-in model is the reference's `model.`)
    sd = {"model.vision_tower." + k: v for k, v in tower_sd.items()}
    sd.update({"model.mm_projector." + k: v for k, v in fx.projector_state_dict(128).items()})
    want = [l.strip() for l in open(os.path.join(golden_dir, "llava_model_keys.txt")) if l.strip()]
    assert sorted(sd) == sorted(want)
    model.load_state_dict({k[len("model."):]: v for k, v in sd.items()}, strict=True)
    assert tower.hidden_size == 3072 and tower.num_patches == 16 and tower.num_patches_per_side == 4
    assert llava_arch.LlavaMetaForCausalLM.encode_images is pkg.EncodeImagesMixin.encode_images
    x = fx.synthetic_images(2, 256)
    with torch.inference_mode(), pytest.raises(pkg.FvhdError):      # dispatches to the library: CPU host -> loud failure
        model.encode_images(x)
    if torch.cuda.is_available():
        model.to(device="cuda", dtype=torch.bfloat16)
        with torch.inference_mode():
            feats = model.encode_images(x.to("cuda"))
        assert tuple(feats.shape) == (2, 16, 128)

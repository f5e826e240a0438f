"""SDLoraManager (SURVEY.md section 2 #10): named LoRA sets on a Stable Diffusion UNet.

Stand-alone behaviour (names, scales, removal, the "already exists" / "subset" assertions) and the same operations as
recorded on the reference (tests/golden/structure.json.xz): the same module tree, the same exported weight keys and the
same checkpoint-key ordering."""

import pytest
import torch

import refiners_b200.fluxion.layers as fl
from refiners_b200.foundationals.latent_diffusion import SD1UNet
from refiners_b200.foundationals.latent_diffusion.lora import SDLoraManager

BANNED = {"TimestepEncoder", "ResidualBlock", "Downsample", "Upsample"}


class Holder:
    """The three attributes of a LatentDiffusionModel the manager touches."""

    def __init__(self, unet, encoder=None):
        self.unet, self.clip_text_encoder = unet, encoder
        self.device, self.dtype = torch.device("meta"), torch.float32


def checkpoint(unet, layers_module) -> dict[str, torch.Tensor]:
    """A complete CivitAI-style LoRA state dict for the transformer-block Linears of ``unet`` (rank 4, meta tensors)."""
    tensors, i = {}, 0
    for lin, parent in unet.walk(layers_module.Linear):
        if {type(p).__name__ for p in [*parent.get_parents(), parent]} & BANNED:
            continue
        tensors[f"lora_unet_{i:04d}_x.down.weight"] = torch.empty(4, lin.in_features, device="meta")
        tensors[f"lora_unet_{i:04d}_x.up.weight"] = torch.empty(lin.out_features, 4, device="meta")
        i += 1
    return tensors


def test_manager_add_scale_remove():
    unet = SD1UNet(4, device="meta")
    manager = SDLoraManager(Holder(unet))
    pristine = repr(unet)
    tensors = checkpoint(unet, fl)
    assert manager.names == [] and manager.scales == {}
    manager.add_loras("style", tensors=tensors, scale=0.4)
    manager.add_loras("subject", tensors)
    assert set(manager.names) == {"style", "subject"} and manager.scales == {"style": 0.4, "subject": 1.0}
    assert len(manager.lora_adapters) == len(tensors) // 2 and len(manager.get_loras_by_name("style")) == len(tensors) // 2
    with pytest.raises(AssertionError, match="already exists"):
        manager.add_loras("style", tensors=tensors)
    with pytest.raises(AssertionError, match="subset"):
        manager.update_scales({"nobody": 1.0})
    manager.set_scale("style", 0.9)
    assert manager.get_scale("style") == 0.9
    exported = manager.get_lora_weights("style")
    assert len(exported) == len(tensors) and all(k.endswith((".down.weight", ".up.weight")) for k in exported)
    manager.remove_loras("style")
    assert manager.names == ["subject"]
    manager.remove_all()
    assert manager.names == [] and repr(unet) == pristine


def test_manager_matches_the_reference():
    from tests.test_reference_structure import recorded_values

    for key, want in recorded_values("lora_manager.sort_keys").items():
        assert list(SDLoraManager.sort_keys(key)) == want, key
    ours = SD1UNet(4, device="meta")
    mine = SDLoraManager(Holder(ours))
    tensors = checkpoint(ours, fl)
    assert list(tensors) == recorded_values("lora_manager.checkpoint_keys")

    def tree(unet):  # the Lambda line prints a function signature whose annotations differ (jaxtyping): not structure
        return [line for line in repr(unet).splitlines() if "Lambda(compute_sinusoidal_embedding" not in line]

    for name, scale in (("a", 0.4), ("b", 1.0)):
        mine.add_loras(name, tensors=tensors, scale=scale)
    assert sorted(mine.names) == recorded_values("lora_manager.names") and mine.scales == recorded_values("lora_manager.scales")
    assert list(mine.get_lora_weights("a")) == recorded_values("lora_manager.weights_a")
    assert tree(ours) == recorded_values("lora_manager.tree.added")
    mine.remove_loras("a")
    assert tree(ours) == recorded_values("lora_manager.tree.removed_a")
    mine.remove_all()
    assert tree(ours) == recorded_values("lora_manager.tree.removed_all")

"""Structure parity against the reference, from its recorded surface (tests/golden/structure.json.xz, written by
oracle/pin_against_reference.py --only-surface).

Every model of the hot path is built on the meta device from refiners_b200 and must agree with the reference's
recording on the full `repr()` tree (class names, tags, argument echo: what the reference's own structure tests
assert on, e.g. tests/adapters/test_ip_adapter.py:29-41) and on the state-dict contract (same keys in the same
order, same shapes), before and after adapter injection."""

import functools
import hashlib
import json
import lzma
import re
from pathlib import Path

import pytest
import torch

GOLDEN = Path(__file__).parent / "golden"


@functools.cache
def recorded() -> dict:
    """{"trees": {name: {"tree", "contract"}}, "values": {name: json value or tensor digest}} as the reference produced them."""
    with lzma.open(GOLDEN / "structure.json.xz", "rt", encoding="utf-8") as f:
        return json.load(f)


def recorded_values(name: str):
    return recorded()["values"][name]


def digest(t: torch.Tensor) -> str:
    """SHA-256 of dtype, shape and bytes: equal digests mean bit-identical tensors."""
    t = t.detach().cpu().contiguous()
    return hashlib.sha256(f"{t.dtype} {tuple(t.shape)} ".encode() + t.reshape(-1).view(torch.uint8).numpy().tobytes()).hexdigest()


def contract(module):
    return [(k, tuple(v.shape)) for k, v in module.state_dict().items()]


def tree(module) -> str:
    """repr() with the signature echo of Lambda layers reduced to the function name: the reference annotates its
    helper functions with jaxtyping shapes, which is typing style, not structure."""
    return re.sub(r"Lambda\((\w+)\(.*$", r"Lambda(\1)", repr(module), flags=re.MULTILINE)


def same(mine, name: str) -> None:
    """``mine`` has the state-dict contract and the tree the reference recorded under ``name``."""
    want = recorded()["trees"][name]
    assert contract(mine) == [(k, tuple(s)) for k, s in want["contract"]], name
    assert tree(mine) == want["tree"], name


def same_tree(mine, name: str) -> None:
    assert tree(mine) == recorded()["trees"][name]["tree"], name


def test_sd1_unet_and_controlnet():
    from refiners_b200.foundationals.latent_diffusion.stable_diffusion_1 import SD1ControlnetAdapter, SD1UNet

    mine = SD1UNet(4, device="meta")
    same(mine, "sd1.unet")
    a = SD1ControlnetAdapter(mine, name="canny", scale=0.9).inject()
    same(mine, "sd1.unet.controlnet")
    same_tree(a, "sd1.controlnet")
    a.eject()
    same(mine, "sd1.unet.controlnet_ejected")


def test_sdxl_unet_control_lora_and_ip_adapter():
    from refiners_b200.foundationals.latent_diffusion import SDXLUNet
    from refiners_b200.foundationals.latent_diffusion.image_prompt import SDXLIPAdapter
    from refiners_b200.foundationals.latent_diffusion.stable_diffusion_xl.control_lora import ControlLoraAdapter

    mine = SDXLUNet(4, device="meta")
    same(mine, "sdxl.unet")
    a = ControlLoraAdapter("canny", mine, scale=0.8).inject()
    same(mine, "sdxl.unet.control_lora")
    a.eject()
    same(mine, "sdxl.unet.control_lora_ejected")
    ia = SDXLIPAdapter(mine, scale=0.5)
    ia.inject()
    same(mine, "sdxl.unet.ip_adapter")
    assert contract(ia.image_proj) == [(k, tuple(s)) for k, s in recorded()["trees"]["sdxl.ip_adapter.image_proj"]["contract"]]
    ia.eject()
    same(mine, "sdxl.unet.ip_adapter_ejected")


def keyed(module, seed: int):
    """The module with the keyed weights the reference ran with when the fixture was recorded."""
    from oracle.weights import keyed_state_dict

    module.load_state_dict(keyed_state_dict({k: tuple(v.shape) for k, v in module.state_dict().items()}, seed=seed))
    return module


def test_ip_adapter_plus_perceiver_resampler():
    """fine_grained=True: the 16-token PerceiverResampler image projection, structure and numbers (same weights)."""
    from refiners_b200.foundationals.latent_diffusion import SDXLUNet
    from refiners_b200.foundationals.latent_diffusion.image_prompt import SDXLIPAdapter
    from refiners_b200.foundationals.latent_diffusion.perceiver import PerceiverResampler

    ia = SDXLIPAdapter(SDXLUNet(4, device="meta"), fine_grained=True)
    assert isinstance(ia.image_proj, PerceiverResampler)
    same(ia.image_proj, "perceiver.image_proj")
    cfg = dict(latents_dim=64, num_attention_layers=2, num_attention_heads=4, head_dim=16, num_tokens=5, input_dim=48, output_dim=40)
    mine = keyed(PerceiverResampler(**cfg), 31)
    x = torch.randn(3, 11, 48, generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        assert digest(mine(x)) == recorded_values("perceiver.y")


def test_clip_image_encoder_and_image_embedding():
    """CLIP vision tower (structure of H; numbers on a tiny tower with the reference's weights) and the IP-Adapter's
    once-per-prompt path image -> context tensor, including weights and token concatenation."""
    import refiners_b200.fluxion.layers as fl
    from refiners_b200.foundationals.clip import CLIPImageEncoder, CLIPImageEncoderH
    from refiners_b200.foundationals.latent_diffusion import CrossAttentionBlock2d
    from refiners_b200.foundationals.latent_diffusion.image_prompt import ImageProjection, IPAdapter

    mine_h = CLIPImageEncoderH(device="meta")
    same(mine_h, "clip.image_encoder_h")
    same(IPAdapter.convert_to_grid_features(mine_h), "clip.image_encoder_h.grid")

    cfg = dict(image_size=32, embedding_dim=48, output_dim=24, patch_size=8, num_layers=2, num_attention_heads=3, feedforward_dim=96)
    block = dict(channels=64, context_embedding_dim=40, context_key="ctx", num_attention_heads=2, use_linear_projection=True)
    enc_m = keyed(CLIPImageEncoder(**cfg), 32)
    proj_m = keyed(ImageProjection(clip_image_embedding_dim=24, clip_text_embedding_dim=40), 33)
    ip_m = IPAdapter(fl.Chain(CrossAttentionBlock2d(**block)), enc_m, proj_m)
    images = torch.randn(3, 3, 32, 32, generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        assert digest(enc_m(images)) == recorded_values("clip.encoded")
        for i, kwargs in enumerate(({}, {"weights": [1.0, 0.5, 2.0]}, {"concat_batches": False})):
            assert digest(ip_m.compute_clip_image_embedding(images, **kwargs)) == recorded_values(f"clip.embedding.{i}"), kwargs


def test_lora_adapters_on_cross_attention():
    import refiners_b200.fluxion.layers as fl
    from refiners_b200.fluxion.adapters import LinearLora, LoraAdapter
    from refiners_b200.foundationals.latent_diffusion import CrossAttentionBlock2d

    kw = dict(channels=64, context_embedding_dim=48, context_key="ctx", num_attention_heads=2, num_attention_layers=2,
              use_linear_projection=True, device="meta")
    mine = fl.Chain(CrossAttentionBlock2d(**kw))
    same(mine, "lora.block")
    for lin, parent in list(mine.walk(fl.Linear, recurse=True)):
        loras = [LinearLora(f"l{j}", in_features=lin.in_features, out_features=lin.out_features, rank=4, scale=s, device="meta")
                 for j, s in enumerate((1.0, 1.4))]
        LoraAdapter(lin, *loras).inject(parent)
    same(mine, "lora.block.loras")


def test_sam_vit_h():
    from refiners_b200.foundationals.segment_anything import SAMViTH

    same(SAMViTH(device="meta"), "sam.vit_h")


def test_vae():
    from refiners_b200.foundationals.latent_diffusion.auto_encoder import LatentDiffusionAutoencoder

    same(LatentDiffusionAutoencoder(device="meta"), "vae")


@pytest.mark.parametrize("name", ["DINOv2_small", "DINOv2_base_reg", "DINOv2_large", "DINOv2_giant_reg"])
def test_dinov2(name):
    import refiners_b200.foundationals.dinov2 as mine

    same(getattr(mine, name)(device="meta"), f"dinov2.{name}")


def test_solver_tables():
    from refiners_b200.foundationals.latent_diffusion import DDIM, Euler

    for tag, mine in (("euler", Euler(num_inference_steps=30)), ("ddim", DDIM(num_inference_steps=20))):
        for table in ("timesteps", "cumulative_scale_factors", "noise_std"):
            assert digest(getattr(mine, table)) == recorded_values(f"solver.{tag}.{table}"), (tag, table)

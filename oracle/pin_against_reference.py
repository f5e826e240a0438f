"""Pin the oracle against the REAL reference and (re)generate tests/golden/*.safetensors.

Run only where /root/reference is mounted (the build container):

    python oracle/pin_against_reference.py            # check + write fixtures
    python oracle/pin_against_reference.py --check    # check only

For every case the reference's own modules (imported unmodified from /root/reference/src) are
evaluated in fp32 on the CPU; the oracle restatement must agree within 1e-5 * max|ref|, and the
reference's inputs/outputs (plus weights, for the small cases) are stored as fixtures.  The GPU
box has no /root/reference: tests there read only the committed fixtures.
TEST INFRASTRUCTURE - see oracle/__init__.py.
"""

from __future__ import annotations

import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
REF_SRC = Path("/root/reference/src")
GOLDEN = ROOT / "tests" / "golden"


def _import_reference():
    if not REF_SRC.exists():
        raise SystemExit("/root/reference is not mounted here: nothing to pin against")
    stub = Path("/tmp/rb200_refstub")
    meta = stub / "refiners-0.0.0.dist-info"
    meta.mkdir(parents=True, exist_ok=True)
    (meta / "METADATA").write_text("Metadata-Version: 2.1\nName: refiners\nVersion: 0.0.0\nRequires-Dist: torch\n")
    for p in (str(REF_SRC), str(stub), str(ROOT)):
        if p not in sys.path:
            sys.path.insert(0, p)
    import refiners.fluxion.layers as rfl  # noqa: F401

    return rfl


def _close(name: str, got: torch.Tensor, want: torch.Tensor, rel: float = 1e-5) -> None:
    err = (got - want).abs().max().item()
    tol = rel * max(want.abs().max().item(), 1e-3)
    status = "ok " if err <= tol else "FAIL"
    print(f"  [{status}] {name}: max abs diff {err:.3e} (tol {tol:.3e})")
    if err > tol:
        raise SystemExit(f"oracle disagrees with the reference on {name}")


def control_lora_test_weights() -> dict[str, torch.Tensor]:
    """A small synthetic ControlLora checkpoint (shape conventions of control_lora.py:319-411): rank-4
    LoRAs on three shared leaves; zero-convs and the condition encoder keep their (keyed) weights."""
    gen = torch.Generator().manual_seed(99)
    targets = {
        "DownBlocks.Chain_5.SDXLCrossAttention.Chain_2.CrossAttentionBlock_1.Residual_1.SelfAttention.Distribute.Linear_1": (640, 640),
        "DownBlocks.Chain_8.SDXLCrossAttention.Chain_2.CrossAttentionBlock_3.Residual_3.Linear_2": (5120, 1280),
        "MiddleBlock.SDXLCrossAttention.Chain_1.Linear": (1280, 1280),
    }
    sd: dict[str, torch.Tensor] = {}
    for path, (fin, fout) in targets.items():
        sd[f"ControlLora.{path}.down"] = torch.randn(4, fin, generator=gen) * 0.25
        sd[f"ControlLora.{path}.up"] = torch.randn(fout, 4, generator=gen) * 0.05
    return sd


def pin_controlnet(write: bool) -> None:
    """SD 1.5 + ControlNet (stable_diffusion_1/controlnet.py): own generator, own fixture file, so that
    adding it does not disturb the random stream of the other fixtures."""
    _import_reference()
    from refiners.foundationals.latent_diffusion.stable_diffusion_1.controlnet import SD1ControlnetAdapter
    from refiners.foundationals.latent_diffusion.stable_diffusion_1.unet import SD1UNet
    from safetensors.torch import save_file

    from oracle import unet as ounet
    from oracle.weights import keyed_state_dict

    print("SD1UNet + Controlnet")
    gen = torch.Generator().manual_seed(4321)
    g = lambda *s: torch.randn(*s, generator=gen)
    with torch.no_grad():
        unet = SD1UNet(4)
        adapter = SD1ControlnetAdapter(unet, name="canny", scale=0.9, scale_decay=0.825).inject()
        shapes = {k: tuple(v.shape) for k, v in unet.state_dict().items()}
        sdict = keyed_state_dict(shapes, seed=4)
        unet.load_state_dict(sdict)
        x, ts, ctx = g(2, 4, 32, 32), torch.tensor([[500]]), g(2, 77, 768)
        cond = torch.rand(2, 3, 256, 256, generator=gen)
        unet.set_timestep(ts); unet.set_clip_text_embedding(ctx)
        adapter.set_controlnet_condition(cond)
        y = unet(x)
        deltas = ounet.sd1_controlnet(sdict, x, ts, ctx, cond, scale=0.9, scale_decay=0.825)
        _close("SD1UNet + Controlnet", ounet.sd1_unet(sdict, x, ts, ctx, residuals=deltas), y)
        adapter.eject()
        unet.set_timestep(ts); unet.set_clip_text_embedding(ctx)  # contexts are reset after every forward
        y_plain = unet(x)
        plain = {k: v for k, v in sdict.items() if not k.startswith("Controlnet.")}
        _close("SD1UNet after eject", ounet.sd1_unet(plain, x, ts, ctx), y_plain)
    fx = {"cn.x": x, "cn.timestep": ts, "cn.ctx": ctx, "cn.cond": cond, "cn.y": y, "cn.y_plain": y_plain}
    if write:
        GOLDEN.mkdir(parents=True, exist_ok=True)
        save_file({k: v.contiguous() for k, v in fx.items()}, str(GOLDEN / "controlnet.safetensors"))
        print(f"  wrote {GOLDEN / 'controlnet.safetensors'}")


def pin_denoise_step(write: bool) -> None:
    """One full denoising step of the reference's StableDiffusion_1 (LatentDiffusionModel.forward,
    model.py:128-159: contexts, CFG doubling, sigma scaling, UNet, CFG combine, Euler update) on keyed
    weights; own generator and fixture file."""
    _import_reference()
    from refiners.foundationals.latent_diffusion.solvers import Euler
    from refiners.foundationals.latent_diffusion.stable_diffusion_1.model import StableDiffusion_1
    from refiners.foundationals.latent_diffusion.stable_diffusion_1.unet import SD1UNet
    from safetensors.torch import save_file

    from oracle import euler as oeuler
    from oracle import unet as ounet
    from oracle.weights import keyed_state_dict

    print("StableDiffusion_1 denoising step (CFG + Euler)")
    gen = torch.Generator().manual_seed(777)
    g = lambda *s: torch.randn(*s, generator=gen)
    with torch.no_grad():
        unet = SD1UNet(4)
        shapes = {k: tuple(v.shape) for k, v in unet.state_dict().items()}
        sdict = keyed_state_dict(shapes, seed=1)
        unet.load_state_dict(sdict)
        sd = StableDiffusion_1(unet=unet, solver=Euler(num_inference_steps=30))
        x = g(2, 4, 32, 32) * float(sd.solver.init_noise_sigma)
        ctx = g(4, 77, 768)  # unconditional block first, conditional second (model.py:137)
        fx = {"step.x": x, "step.ctx": ctx}
        schedule = oeuler.EulerSchedule(30)
        for step, scale in ((0, 7.5), (7, 5.0), (29, 7.5)):
            y = sd(x, step=step, clip_text_embedding=ctx, condition_scale=scale)
            fx[f"step.y_{step}"] = y
            mine = oeuler.denoise_step(lambda lat, ts: ounet.sd1_unet(sdict, lat, ts, ctx), schedule, x, step, scale)
            _close(f"denoise step {step} (scale {scale})", mine, y)
    if write:
        GOLDEN.mkdir(parents=True, exist_ok=True)
        save_file({k: v.contiguous() for k, v in fx.items()}, str(GOLDEN / "step.safetensors"))
        print(f"  wrote {GOLDEN / 'step.safetensors'}")


def pin_sag(write: bool) -> None:
    """Self-attention guidance: one StableDiffusion_1 step (DDIM, CFG, SAG scale 0.75) on 64x64 latents with keyed
    weights (middle block 8x8 = 64 tokens), the recorded mask included; own generator and fixture file."""
    _import_reference()
    from refiners.foundationals.latent_diffusion.solvers import DDIM
    from refiners.foundationals.latent_diffusion.stable_diffusion_1.model import StableDiffusion_1
    from refiners.foundationals.latent_diffusion.stable_diffusion_1.unet import SD1UNet
    from safetensors.torch import save_file

    from oracle import sag as osag
    from oracle import unet as ounet
    from oracle.weights import keyed_state_dict

    print("StableDiffusion_1 step with self-attention guidance (DDIM)")
    gen = torch.Generator().manual_seed(2210)
    g = lambda *s: torch.randn(*s, generator=gen)
    with torch.no_grad():
        unet = SD1UNet(4)
        sdict = keyed_state_dict({k: tuple(v.shape) for k, v in unet.state_dict().items()}, seed=1)
        unet.load_state_dict(sdict)
        sd = StableDiffusion_1(unet=unet, solver=DDIM(num_inference_steps=30))
        sd.set_self_attention_guidance(enable=True, scale=0.75)
        x, ctx = g(2, 4, 64, 64), g(4, 77, 768)
        fx = {"sag.x": x, "sag.ctx": ctx}
        schedule = osag.DDIMSchedule(30)
        _close("DDIM timesteps", schedule.timesteps.float(), sd.solver.timesteps.float())
        run = lambda lat, ts, guided: ounet.sd1_unet(sdict, lat, ts, ctx if guided else ctx.chunk(2)[0])  # noqa: E731
        for step, scale in ((3, 7.5), (20, 5.0)):
            y = sd(x, step=step, clip_text_embedding=ctx, condition_scale=scale)
            fx[f"sag.y_{step}"] = y
            _close(f"SAG step {step} (scale {scale})", osag.denoise_step(run, schedule, x, step, scale, 0.75), y)
        sd.set_self_attention_guidance(enable=False)
        plain = sd(x, step=3, clip_text_embedding=ctx, condition_scale=7.5)
        print(f"  guidance moves the step-3 result by {float((fx['sag.y_3'] - plain).abs().max()):.3e} (max |y| {float(plain.abs().max()):.3f})")
    if write:
        GOLDEN.mkdir(parents=True, exist_ok=True)
        save_file({k: v.contiguous() for k, v in fx.items()}, str(GOLDEN / "sag.safetensors"))
        print(f"  wrote {GOLDEN / 'sag.safetensors'}")


def pin_t2i(write: bool) -> None:
    """T2I-Adapter: both condition encoders at full width on a 256x256 condition image, and the adapters injected into SD1UNet /
    SDXLUNet (keyed weights, 32x32 latents, scale 0.8); own fixture file (the UNet inputs are keyed, only outputs are stored)."""
    _import_reference()
    from refiners.foundationals.latent_diffusion.stable_diffusion_1.t2i_adapter import SD1T2IAdapter
    from refiners.foundationals.latent_diffusion.stable_diffusion_1.unet import SD1UNet
    from refiners.foundationals.latent_diffusion.stable_diffusion_xl.t2i_adapter import SDXLT2IAdapter
    from refiners.foundationals.latent_diffusion.stable_diffusion_xl.unet import SDXLUNet
    from safetensors.torch import save_file

    from oracle import t2i as ot2i
    from oracle import unet as ounet
    from oracle.cases import keyed_input
    from oracle.weights import keyed_state_dict

    print("T2I-Adapter")
    fx = {}
    with torch.no_grad():
        for tag, unet_cls, adapter_cls, seed in (("sd1", SD1UNet, SD1T2IAdapter, 1), ("sdxl", SDXLUNet, SDXLT2IAdapter, 2)):
            unet = unet_cls(4)
            usd = keyed_state_dict({k: tuple(v.shape) for k, v in unet.state_dict().items()}, seed=seed)
            unet.load_state_dict(usd)
            adapter = adapter_cls(unet, name="depth", scale=0.8)
            esd = keyed_state_dict({k: tuple(v.shape) for k, v in adapter.condition_encoder.state_dict().items()}, seed=31)
            adapter.condition_encoder.load_state_dict(esd)
            adapter.inject()
            condition = keyed_input(f"t2i.{tag}.condition", (1, 3, 256, 256))
            features = adapter.compute_condition_features(condition)
            mine = ot2i.condition_encoder(esd, condition, xl=(tag == "sdxl"))
            for n, (a, b) in enumerate(zip(mine, features)):
                _close(f"{tag} condition feature {n} {tuple(b.shape)}", a, b)
            adapter.set_condition_features(features)
            x, ts = keyed_input(f"t2i.{tag}.x", (1, 4, 32, 32)), torch.tensor([601.0])
            unet.set_timestep(ts)
            if tag == "sd1":
                ctx = keyed_input("t2i.sd1.ctx", (1, 77, 768))
                unet.set_clip_text_embedding(ctx)
                y = unet(x)
                _close("SD1UNet + T2I-Adapter", ounet.sd1_unet(usd, x, ts, ctx, t2i=(mine, 0.8)), y)
            else:
                ctx, pooled = keyed_input("t2i.sdxl.ctx", (1, 77, 2048)), keyed_input("t2i.sdxl.pooled", (1, 1280))
                ids = torch.tensor([[1024.0, 1024, 0, 0, 1024, 1024]])
                unet.set_clip_text_embedding(ctx); unet.set_pooled_text_embedding(pooled); unet.set_time_ids(ids)
                y = unet(x)
                _close("SDXLUNet + T2I-Adapter", ounet.sdxl_unet(usd, x, ts, ctx, pooled, ids, t2i=(mine, 0.8)), y)
            fx[f"{tag}.y"] = y
            fx[f"{tag}.feature_3"] = features[3]  # the coarsest map; the others are re-derived by the (pinned) oracle in the tests
    if write:
        save_file({k: v.contiguous() for k, v in fx.items()}, str(GOLDEN / "t2i.safetensors"))
        print(f"  wrote {GOLDEN / 't2i.safetensors'}")


def pin_style_aligned(write: bool) -> None:
    """StyleAligned on SD1UNet and SDXLUNet (keyed weights, guidance batch of 2 x 2 images at 32x32 latents, scale 0.7); own
    fixture file (inputs are keyed, only outputs are stored)."""
    _import_reference()
    from refiners.foundationals.latent_diffusion.stable_diffusion_1.unet import SD1UNet
    from refiners.foundationals.latent_diffusion.stable_diffusion_xl.unet import SDXLUNet
    from refiners.foundationals.latent_diffusion.style_aligned import StyleAlignedAdapter
    from safetensors.torch import save_file

    from oracle import unet as ounet
    from oracle.cases import keyed_input
    from oracle.weights import keyed_state_dict

    print("StyleAligned")
    fx = {}
    with torch.no_grad():
        for tag, unet_cls, seed, width in (("sd1", SD1UNet, 1, 768), ("sdxl", SDXLUNet, 2, 2048)):
            unet = unet_cls(4)
            usd = keyed_state_dict({k: tuple(v.shape) for k, v in unet.state_dict().items()}, seed=seed)
            unet.load_state_dict(usd)
            StyleAlignedAdapter(unet, scale=0.7).inject()
            x, ts = keyed_input(f"style.{tag}.x", (4, 4, 32, 32)), torch.tensor([601.0])
            ctx = keyed_input(f"style.{tag}.ctx", (4, 77, width))
            unet.set_timestep(ts); unet.set_clip_text_embedding(ctx)
            ounet.style_aligned_scale = 0.7
            try:
                if tag == "sd1":
                    y = unet(x)
                    mine = ounet.sd1_unet(usd, x, ts, ctx)
                else:
                    pooled, ids = keyed_input("style.sdxl.pooled", (4, 1280)), torch.tensor([[1024.0, 1024, 0, 0, 1024, 1024]] * 4)
                    unet.set_pooled_text_embedding(pooled); unet.set_time_ids(ids)
                    y = unet(x)
                    mine = ounet.sdxl_unet(usd, x, ts, ctx, pooled, ids)
            finally:
                ounet.style_aligned_scale = None
            _close(f"{tag} UNet + StyleAligned", mine, y)
            fx[f"{tag}.y"] = y
    if write:
        save_file({k: v.contiguous() for k, v in fx.items()}, str(GOLDEN / "style_aligned.safetensors"))
        print(f"  wrote {GOLDEN / 'style_aligned.safetensors'}")


def pin_vae(write: bool) -> None:
    """LatentDiffusionAutoencoder.encode / decode (auto_encoder.py:305-331) on keyed weights; own fixture file."""
    _import_reference()
    from refiners.foundationals.latent_diffusion.auto_encoder import LatentDiffusionAutoencoder
    from safetensors.torch import save_file

    from oracle import vae as ovae
    from oracle.weights import keyed_state_dict

    print("LatentDiffusionAutoencoder")
    gen = torch.Generator().manual_seed(2468)
    with torch.no_grad():
        lda = LatentDiffusionAutoencoder()
        shapes = {k: tuple(v.shape) for k, v in lda.state_dict().items()}
        sdict = keyed_state_dict(shapes, seed=5)
        lda.load_state_dict(sdict)
        z = torch.randn(2, 4, 12, 16, generator=gen)
        image = torch.rand(1, 3, 72, 56, generator=gen) * 2 - 1
        x = lda.decode(z)
        lat = lda.encode(image)
        _close("VAE decode", ovae.decode(sdict, z), x)
        _close("VAE encode", ovae.encode(sdict, image), lat)
    fx = {"vae.z": z, "vae.decoded": x, "vae.image": image, "vae.encoded": lat}
    if write:
        GOLDEN.mkdir(parents=True, exist_ok=True)
        save_file({k: v.contiguous() for k, v in fx.items()}, str(GOLDEN / "vae.safetensors"))
        print(f"  wrote {GOLDEN / 'vae.safetensors'}")


def pin_vae_tiled(write: bool) -> None:
    """Tiled VAE inference (auto_encoder.py:209-279, 411-621): a 224x160 image in 128x96 tiles blended over 32 pixels
    (2 x 2 tiles), GroupNorm statistics frozen from the resized image; own generator and fixture file."""
    _import_reference()
    import numpy as np
    from PIL import Image
    from refiners.fluxion.utils import image_to_tensor
    from refiners.foundationals.latent_diffusion.auto_encoder import LatentDiffusionAutoencoder
    from safetensors.torch import save_file

    from oracle import vae as ovae
    from oracle.weights import keyed_state_dict

    print("LatentDiffusionAutoencoder, tiled inference")
    pixels = (np.random.default_rng(3).random((160, 224, 3)) * 255).astype(np.uint8)
    image = Image.fromarray(pixels)
    tile, blending = (128, 96), 32  # (width, height)
    with torch.no_grad():
        lda = LatentDiffusionAutoencoder()
        sdict = keyed_state_dict({k: tuple(v.shape) for k, v in lda.state_dict().items()}, seed=5)
        lda.load_state_dict(sdict)
        with lda.tiled_inference(image, tile_size=tile, blending=blending):
            latents = lda.tiled_image_to_latents(image)
            decoded = lda._tiled_decode(latents, lda._tile_size, blending)
        full, small = image_to_tensor(image), image_to_tensor(image.resize(tile))
        ovae.frozen_stats = {}
        try:
            ovae.capture_statistics(sdict, full, small)
            mine_lat = ovae.tiled(sdict, ovae.encode, 2 * full - 1, (20, 28), (96, 128), blending, 8, 1, 4)
            mine_dec = ovae.tiled(sdict, ovae.decode, latents, (20, 28), (96, 128), blending, 1, 8, 3)
        finally:
            ovae.frozen_stats = None
        _close("tiled encode", mine_lat, latents)
        _close("tiled decode", mine_dec, decoded)
    fx = {"tiled.pixels": torch.from_numpy(pixels), "tiled.small": (small * 255).round().to(torch.uint8), "tiled.latents": latents,
          "tiled.decoded": decoded}
    if write:
        save_file({k: v.contiguous() for k, v in fx.items()}, str(GOLDEN / "vae_tiled.safetensors"))
        print(f"  wrote {GOLDEN / 'vae_tiled.safetensors'}")


def pin_dinov2(write: bool) -> None:
    """DINOv2 ViT (dinov2/vit.py:289-413): the published small model at 224x224, and a tiny register + SwiGLU
    configuration on a non-square input that exercises the antialiased bicubic resize of the positions."""
    _import_reference()
    import refiners.fluxion.layers as rfl
    from refiners.foundationals.dinov2 import DINOv2_small, ViT
    from safetensors.torch import save_file

    from oracle import dinov2 as odino
    from oracle.weights import keyed_state_dict

    print("DINOv2 ViT")
    gen = torch.Generator().manual_seed(1357)
    fx = {}
    with torch.no_grad():
        small = DINOv2_small()
        sd = keyed_state_dict({k: tuple(v.shape) for k, v in small.state_dict().items()}, seed=6)
        small.load_state_dict(sd)
        x = torch.randn(2, 3, 224, 224, generator=gen)
        y = small(x)
        _close("DINOv2_small", odino.vit(sd, x, patch_size=14, num_layers=12, num_heads=6), y)
        fx.update({"small.x": x, "small.y": y})
        tiny_cfg = dict(embedding_dim=64, patch_size=4, image_size=16, num_layers=2, num_heads=2, num_registers=3,
                        feedforward_dim=96, interpolate_antialias=True)
        tiny = ViT(activation=rfl.GLU(rfl.SiLU()), **tiny_cfg)
        sd = keyed_state_dict({k: tuple(v.shape) for k, v in tiny.state_dict().items()}, seed=7)
        tiny.load_state_dict(sd)
        x = torch.randn(3, 3, 24, 20, generator=gen)
        y = tiny(x)
        _close("ViT tiny (registers, SwiGLU, 6x5 grid)", odino.vit(sd, x, patch_size=4, num_layers=2, num_heads=2, num_registers=3,
                                                                    swiglu=True, interpolate_antialias=True), y)
        fx.update({"tiny.x": x, "tiny.y": y})
    if write:
        GOLDEN.mkdir(parents=True, exist_ok=True)
        save_file({k: v.contiguous() for k, v in fx.items()}, str(GOLDEN / "dinov2.safetensors"))
        print(f"  wrote {GOLDEN / 'dinov2.safetensors'}")


def pin_clip(write: bool) -> None:
    """CLIP vision towers (clip/image_encoder.py): ViT-H/14 - the IP-Adapter's image encoder (d = 80, 257 tokens) - and a
    tiny configuration (d = 16, 17 tokens), keyed weights, own fixture file."""
    _import_reference()
    from refiners.foundationals.clip.image_encoder import CLIPImageEncoder, CLIPImageEncoderH
    from safetensors.torch import save_file

    from oracle import clip as oclip
    from oracle.cases import keyed_input
    from oracle.weights import keyed_state_dict

    print("CLIP image encoders")
    fx = {}
    with torch.no_grad():
        big = CLIPImageEncoderH()
        sd = keyed_state_dict({k: tuple(v.shape) for k, v in big.state_dict().items()}, seed=9)
        big.load_state_dict(sd)
        x = keyed_input("clip.h.image", (2, 3, 224, 224))
        y = big(x)
        _close("CLIPImageEncoderH", oclip.image_encoder(sd, x, patch_size=14, num_layers=32, num_heads=16), y, rel=2e-5)
        fx["h.y"] = y
        tiny_cfg = dict(image_size=32, embedding_dim=32, output_dim=16, patch_size=8, num_layers=2, num_attention_heads=2, feedforward_dim=64)
        tiny = CLIPImageEncoder(**tiny_cfg)
        sd = keyed_state_dict({k: tuple(v.shape) for k, v in tiny.state_dict().items()}, seed=10)
        tiny.load_state_dict(sd)
        x = keyed_input("clip.tiny.image", (3, 3, 32, 32))
        y = tiny(x)
        _close("CLIPImageEncoder tiny", oclip.image_encoder(sd, x, patch_size=8, num_layers=2, num_heads=2), y)
        fx["tiny.y"] = y
    if write:
        GOLDEN.mkdir(parents=True, exist_ok=True)
        save_file({k: v.contiguous() for k, v in fx.items()}, str(GOLDEN / "clip.safetensors"))
        print(f"  wrote {GOLDEN / 'clip.safetensors'}")


PROMPTS = ["a photo of a cat", "", "An astronaut riding a horse on Mars, 4k, highly-detailed!!"]


def pin_clip_text(write: bool) -> None:
    """CLIP text towers: CLIPTextEncoderL (SD 1.5's prompt encoder) and SDXL's DoubleTextEncoder (L + bigG + pooling) on three
    prompts, keyed weights; the token ids are stored too, so the GPU box needs no vocabulary file.  Own fixture file."""
    _import_reference()
    from refiners.foundationals.clip.text_encoder import CLIPTextEncoderL
    from refiners.foundationals.latent_diffusion.stable_diffusion_xl.text_encoder import DoubleTextEncoder
    from safetensors.torch import save_file

    from oracle import clip as oclip
    from oracle.weights import keyed_state_dict

    print("CLIP text encoders")
    fx = {}
    with torch.no_grad():
        tower = CLIPTextEncoderL()
        sd = keyed_state_dict({k: tuple(v.shape) for k, v in tower.state_dict().items()}, seed=21)
        tower.load_state_dict(sd)
        tokens = tower[0](PROMPTS)
        y = tower(PROMPTS)
        _close("CLIPTextEncoderL", oclip.text_encoder(sd, tokens, num_layers=12, heads=12, quick_gelu=True), y)
        fx.update({"l.tokens": tokens, "l.y": y})
        del tower
        double = DoubleTextEncoder()
        sd = keyed_state_dict({k: tuple(v.shape) for k, v in double.state_dict().items()}, seed=22)
        double.load_state_dict(sd)
        from refiners.foundationals.clip.tokenizer import CLIPTokenizer

        tokens_g = CLIPTokenizer(pad_token_id=0)(PROMPTS)
        embedding, pooled = double(PROMPTS)
        towers = oclip.split_double_text_encoder(sd)
        mine = oclip.double_text_encoder(*towers, tokens, tokens_g)
        _close("DoubleTextEncoder embedding", mine[0], embedding)
        _close("DoubleTextEncoder pooled", mine[1], pooled)
        fx.update({"xl.tokens_g": tokens_g, "xl.embedding": embedding, "xl.pooled": pooled})
    if write:
        save_file({k: v.contiguous() for k, v in fx.items()}, str(GOLDEN / "clip_text.safetensors"))
        print(f"  wrote {GOLDEN / 'clip_text.safetensors'}")


def pin_full_size(write: bool) -> None:
    """BASELINE-size cases (oracle/cases.py): SDXLUNet at 128x128 latents plain (config 2), with 700 LoRA
    adapters + IP-Adapter (config 3), with ControlLora (config 4), one full StableDiffusion_XL step with CFG +
    Euler at three steps (A17) and the SAM ViT-H encoder on a 1024^2 image (config 5).  Inputs and adapter
    weights are keyed (regenerated anywhere); only the reference's outputs are stored.
    ``--cases=cfg2,step,cfg3,cfg4,cfg5`` re-records a subset and merges it into the existing file."""
    _import_reference()
    import gc
    import time

    from safetensors.torch import load_file, save_file

    from oracle import cases
    from oracle import euler as oeuler
    from oracle import sam as osam
    from oracle import unet as ounet

    api = cases.reference_api()
    path = GOLDEN / "full_size.safetensors"
    fx: dict[str, torch.Tensor] = load_file(str(path)) if path.exists() else {}
    wanted = next((a.split("=", 1)[1].split(",") for a in sys.argv if a.startswith("--cases=")), ["cfg2", "step", "cfg3", "cfg4", "cfg5"])
    t0 = time.time()

    def save() -> None:
        print(f"  ({time.time() - t0:.0f} s)")
        if write:
            GOLDEN.mkdir(parents=True, exist_ok=True)
            save_file({k: v.contiguous() for k, v in fx.items()}, str(path))
            print(f"  wrote {path}: {sorted(fx)}")

    with torch.no_grad():
        base = cases.sdxl_base_weights(api) if set(wanted) - {"cfg5"} else {}
        print(f"full size: base weights ready ({time.time() - t0:.0f} s)")

        if {"cfg2", "step", "cfg3"} & set(wanted):
            unet = cases.build_sdxl(api, base)
            if "cfg2" in wanted:
                inp = cases.sdxl_inputs("cfg2", 2)
                cases.set_sdxl_contexts(unet, inp)
                y = unet(inp["x"])
                fx["cfg2.y"] = y
                _close("config 2: SDXLUNet 128x128 B=2", ounet.sdxl_unet(base, inp["x"], inp["timestep"], inp["ctx"], inp["pooled"], inp["time_ids"]), y)
                save()
            if "step" in wanted:  # StableDiffusion_XL step (A17) on the plain UNet
                sdxl = api.StableDiffusion_XL(unet=unet, solver=api.Euler(num_inference_steps=30))
                sin = cases.step_inputs()
                x0 = sin["x"] * float(sdxl.solver.init_noise_sigma)
                schedule = oeuler.EulerSchedule(30)
                for step, scale in cases.STEP_CASES:
                    y = sdxl(x0, step=step, clip_text_embedding=sin["ctx"], pooled_text_embedding=sin["pooled"], time_ids=sin["time_ids"],
                             condition_scale=scale)
                    fx[f"step.y_{step}"] = y
                    mine = oeuler.denoise_step(
                        lambda lat, ts: ounet.sdxl_unet(base, lat, ts, sin["ctx"], sin["pooled"], sin["time_ids"]), schedule, x0, step, scale)
                    _close(f"StableDiffusion_XL step {step} (scale {scale})", mine, y)
                del sdxl
                save()
            if "cfg3" in wanted:  # adapters injected into the same UNet
                inp = cases.sdxl_inputs("cfg3", 2)
                ip, extra = cases.attach_config3(api, unet, 2)
                assert extra["n_lora_adapters"] == 700, extra["n_lora_adapters"]
                cases.set_sdxl_contexts(unet, inp)
                y = unet(inp["x"])
                fx["cfg3.y"] = y
                w3 = ounet.Weights(base, loras=extra["loras"], ip=extra["ip"], ip_scale=extra["ip_scale"], ip_embedding=extra["ip_embedding"])
                _close("config 3: + 700 LoRA adapters + IP-Adapter", ounet.sdxl_unet(w3, inp["x"], inp["timestep"], inp["ctx"], inp["pooled"], inp["time_ids"]), y)
                del ip, w3, extra
                save()
            del unet
            gc.collect()

        if "cfg4" in wanted:
            inp = cases.sdxl_inputs("cfg4", 2)
            unet = cases.build_sdxl(api, base)
            adapter, extra = cases.attach_config4(api, unet, 2)
            cases.set_sdxl_contexts(unet, inp)
            y = unet(inp["x"])
            fx["cfg4.y"] = y
            wc = ounet.Weights(base, loras=extra["loras"])
            args = (inp["timestep"], inp["ctx"], inp["pooled"], inp["time_ids"])
            deltas = ounet.sdxl_control_lora(wc, extra["own"], inp["x"], *args, extra["condition"], scale=extra["scale"])
            _close(f"config 4: + ControlLora ({extra['n_loras']} LoRAs)", ounet.sdxl_unet(base, inp["x"], *args, residuals=deltas), y)
            del unet, adapter, wc, extra, deltas
            save()
        del base
        gc.collect()

        if "cfg5" in wanted:
            sam, sd = cases.build_sam(api)
            img = cases.sam_inputs()
            y = sam(img)
            fx["cfg5.y"] = y
            _close("config 5: SAMViTH 1024^2", osam.sam_vit(sd, img, num_layers=32, heads=16, global_indices=(7, 15, 23, 31)), y)
            save()


def main(write: bool) -> None:
    rfl = _import_reference()
    from safetensors.torch import save_file

    from oracle import euler as oeuler
    from oracle import ops, sam as osam, unet as ounet
    from oracle.weights import keyed_state_dict

    torch.manual_seed(1234)
    g = lambda *s: torch.randn(*s)
    out: dict[str, dict[str, torch.Tensor]] = {}

    with torch.no_grad():
        # ------------------------------------------------------------------ leaf ops
        print("leaf ops")
        fx: dict[str, torch.Tensor] = {}
        lin = rfl.Linear(48, 40)
        x = g(3, 7, 48)
        fx.update({"linear.x": x, "linear.w": lin.weight, "linear.b": lin.bias, "linear.y": lin(x)})
        _close("Linear", ops.linear(x, lin.weight, lin.bias), fx["linear.y"])

        for tag, (k, s, p) in {"3x3": (3, 1, 1), "3x3s2": (3, 2, 1), "1x1": (1, 1, 0)}.items():
            conv = rfl.Conv2d(8, 12, kernel_size=k, stride=s, padding=p)
            x = g(2, 8, 10, 12)
            fx.update({f"conv{tag}.x": x, f"conv{tag}.w": conv.weight, f"conv{tag}.b": conv.bias, f"conv{tag}.y": conv(x)})
            _close(f"Conv2d {tag}", ops.conv2d(x, conv.weight, conv.bias, s, p), fx[f"conv{tag}.y"])

        gn = rfl.GroupNorm(64, 32, eps=1e-6)
        gn.weight.copy_(1 + 0.1 * g(64)); gn.bias.copy_(0.1 * g(64))
        x = g(2, 64, 6, 5) * 2 + 0.3
        fx.update({"gn.x": x, "gn.w": gn.weight, "gn.b": gn.bias, "gn.y": gn(x), "gn_silu.y": rfl.SiLU()(gn(x))})
        _close("GroupNorm", ops.group_norm(x, 32, gn.weight, gn.bias, 1e-6), fx["gn.y"])
        _close("GroupNorm+SiLU", ops.silu(ops.group_norm(x, 32, gn.weight, gn.bias, 1e-6)), fx["gn_silu.y"])

        ln = rfl.LayerNorm(40)
        ln.weight.copy_(1 + 0.1 * g(40)); ln.bias.copy_(0.1 * g(40))
        x = g(2, 9, 40) * 3
        fx.update({"ln.x": x, "ln.w": ln.weight, "ln.b": ln.bias, "ln.y": ln(x)})
        _close("LayerNorm", ops.layer_norm(x, ln.weight, ln.bias, 1e-5), fx["ln.y"])

        ln2 = rfl.LayerNorm2d(16)
        ln2.weight.copy_(1 + 0.1 * g(16)); ln2.bias.copy_(0.1 * g(16))
        x = g(2, 16, 5, 4)
        fx.update({"ln2d.x": x, "ln2d.w": ln2.weight, "ln2d.b": ln2.bias, "ln2d.y": ln2(x)})
        _close("LayerNorm2d", ops.layer_norm_2d(x, ln2.weight, ln2.bias, 1e-6), fx["ln2d.y"])

        x = g(4, 50) * 3
        fx.update({"act.x": x, "silu.y": rfl.SiLU()(x), "gelu.y": rfl.GeLU()(x), "glu.y": rfl.GLU(rfl.GeLU())(x)})
        _close("SiLU", ops.silu(x), fx["silu.y"])
        _close("GeLU", ops.gelu(x), fx["gelu.y"])
        _close("GLU(GeLU)", ops.glu_gelu(x), fx["glu.y"])

        sd = rfl.ScaledDotProductAttention(num_heads=4)
        q, k, v = g(2, 11, 64), g(2, 7, 64), g(2, 7, 64)
        fx.update({"sdpa.q": q, "sdpa.k": k, "sdpa.v": v, "sdpa.y": sd(q, k, v)})
        _close("ScaledDotProductAttention", ops.sdpa(q, k, v, 4), fx["sdpa.y"])
        sdc = rfl.ScaledDotProductAttention(num_heads=2, is_causal=True)
        q = g(1, 9, 32)
        fx.update({"sdpa_causal.q": q, "sdpa_causal.y": sdc(q, q, q)})
        _close("ScaledDotProductAttention causal", ops.sdpa(q, q, q, 2, True), fx["sdpa_causal.y"])

        from refiners.fluxion.adapters.lora import LinearLora, LoraAdapter

        base = rfl.Linear(48, 40)
        holder = rfl.Chain(base)
        l1, l2 = LinearLora("a", in_features=48, out_features=40, rank=4, scale=1.0), LinearLora("b", in_features=48, out_features=40, rank=8, scale=1.4)
        for l in (l1, l2):
            l.up.weight.copy_(0.05 * g(*l.up.weight.shape))
        LoraAdapter(base, l1, l2).inject(holder)
        x = g(5, 48)
        fx.update({"lora.x": x, "lora.w": base.weight, "lora.b": base.bias, "lora.y": holder(x),
                   "lora.down1": l1.down.weight, "lora.up1": l1.up.weight, "lora.down2": l2.down.weight, "lora.up2": l2.up.weight})
        _close("LoraAdapter", ops.lora_linear(x, base.weight, base.bias, [(l1.down.weight, l1.up.weight, 1.0), (l2.down.weight, l2.up.weight, 1.4)]), fx["lora.y"])
        out["ops"] = fx

        # -------------------------------------------------------------------- blocks
        print("blocks (weights stored in the fixture)")
        from refiners.foundationals.latent_diffusion.cross_attention import CrossAttentionBlock2d
        from refiners.foundationals.latent_diffusion.range_adapter import RangeAdapter2d
        from refiners.foundationals.latent_diffusion.unet import ResidualBlock

        fx = {}
        for tag, (cin, cout) in {"res_same": (64, 64), "res_proj": (64, 96)}.items():
            rb = ResidualBlock(cin, cout)
            body = rb.layer("Chain", rfl.Chain)
            RangeAdapter2d(target=body.layer("Conv2d_1", rfl.Conv2d), channels=cout, embedding_dim=32, context_key="timestep_embedding").inject(body)
            top = rfl.Chain(rb)
            temb, x = g(2, 32), g(2, cin, 8, 8)
            top.set_context("range_adapter", {"timestep_embedding": temb})
            y = top(x)
            sdict = {f"{tag}.sd.ResidualBlock.{k}": v for k, v in rb.state_dict().items()}
            fx.update(sdict)
            fx.update({f"{tag}.x": x, f"{tag}.temb": temb, f"{tag}.y": y})
            _close(f"ResidualBlock {cin}->{cout}", ounet.residual_block(rb.state_dict(prefix="ResidualBlock."), "ResidualBlock", x, temb), y)
        for tag, linear_proj in {"xattn_linear": True, "xattn_conv": False}.items():
            ca = CrossAttentionBlock2d(64, context_embedding_dim=48, context_key="ctx", num_attention_heads=2,
                                       num_attention_layers=2, use_bias=False, use_linear_projection=linear_proj)
            ctx, x = g(2, 5, 48), g(2, 64, 4, 6)
            ca.set_context("cross_attention_block", {"ctx": ctx})
            y = ca(x)
            fx.update({f"{tag}.sd.{k}": v for k, v in ca.state_dict().items()})
            fx.update({f"{tag}.x": x, f"{tag}.ctx": ctx, f"{tag}.y": y})
            _close(f"CrossAttentionBlock2d linear={linear_proj}", ounet.cross_attention_2d(ca.state_dict(prefix="X."), "X", x, ctx, 2, 2, linear_proj), y)
        out["blocks"] = fx

        # -------------------------------------------------------------------- solver
        print("Euler solver")
        from refiners.foundationals.latent_diffusion.solvers import Euler

        fx = {}
        ref_solver = Euler(num_inference_steps=30)
        mine = oeuler.EulerSchedule(30)
        x, eps = g(2, 4, 8, 8), g(2, 4, 8, 8)
        fx.update({"euler.sigmas": ref_solver.sigmas, "euler.timesteps": ref_solver.timesteps, "euler.x": x, "euler.eps": eps,
                   "euler.scaled_init": ref_solver.scale_model_input(x, -1), "euler.scaled_7": ref_solver.scale_model_input(x, 7),
                   "euler.step_7": ref_solver(x, predicted_noise=eps, step=7), "euler.step_29": ref_solver(x, predicted_noise=eps, step=29)})
        _close("sigmas", mine.sigmas, ref_solver.sigmas)
        _close("timesteps", mine.timesteps, ref_solver.timesteps)
        _close("scale_model_input(-1)", mine.scale_model_input(x, -1), fx["euler.scaled_init"])
        _close("scale_model_input(7)", mine.scale_model_input(x, 7), fx["euler.scaled_7"])
        _close("update(7)", mine.update(x, eps, 7), fx["euler.step_7"])
        _close("update(29)", mine.update(x, eps, 29), fx["euler.step_29"])
        bf = Euler(num_inference_steps=30).to(dtype=torch.bfloat16)  # how LatentDiffusionModel casts it (model.py:33)
        fx["euler.sigmas_bf16"] = bf.sigmas
        out["euler"] = fx

        # ----------------------------------------------------------------- full UNets
        print("full UNets (weights regenerated from oracle.weights.keyed_state_dict, only I/O stored)")
        from refiners.foundationals.latent_diffusion.stable_diffusion_1.unet import SD1UNet
        from refiners.foundationals.latent_diffusion.stable_diffusion_xl.unet import SDXLUNet

        fx = {}
        unet = SD1UNet(4, device="meta")
        shapes = {k: tuple(v.shape) for k, v in unet.state_dict().items()}
        sdict = keyed_state_dict(shapes, seed=1)
        unet = SD1UNet(4)
        unet.load_state_dict(sdict)
        x, ts, ctx = g(1, 4, 32, 32), torch.tensor([[500]]), g(1, 77, 768)
        unet.set_timestep(ts); unet.set_clip_text_embedding(ctx)
        y = unet(x)
        fx.update({"sd1.x": x, "sd1.timestep": ts, "sd1.ctx": ctx, "sd1.y": y})
        _close("SD1UNet", ounet.sd1_unet(sdict, x, ts, ctx), y)
        del unet, sdict

        unet = SDXLUNet(4, device="meta")
        shapes = {k: tuple(v.shape) for k, v in unet.state_dict().items()}
        sdict = keyed_state_dict(shapes, seed=2)
        unet = SDXLUNet(4)
        unet.load_state_dict(sdict)
        x, ts = g(2, 4, 32, 32), torch.tensor([981.0])
        ctx, pooled = g(2, 77, 2048), g(2, 1280)
        ids = torch.tensor([[1024, 1024, 0, 0, 1024, 1024]]).repeat(2, 1)
        unet.set_timestep(ts); unet.set_clip_text_embedding(ctx); unet.set_pooled_text_embedding(pooled); unet.set_time_ids(ids)
        y = unet(x)
        fx.update({"sdxl.x": x, "sdxl.timestep": ts, "sdxl.ctx": ctx, "sdxl.pooled": pooled, "sdxl.time_ids": ids, "sdxl.y": y})
        _close("SDXLUNet", ounet.sdxl_unet(sdict, x, ts, ctx, pooled, ids), y)
        del unet, sdict
        # SDXL + ControlLora (BASELINE config 4).  Not restated in the oracle: the fixture pins the
        # refiners_b200 mirror directly against the reference's output.
        from refiners.foundationals.latent_diffusion.stable_diffusion_xl.control_lora import ControlLoraAdapter

        unet = SDXLUNet(4)
        adapter = ControlLoraAdapter("canny", unet, scale=0.8).inject()
        lora_sd = control_lora_test_weights()
        ControlLoraAdapter.load_lora_layers("canny", lora_sd, adapter.control_lora)  # zero-convs / encoder keep keyed weights
        shapes = {k: tuple(v.shape) for k, v in unet.state_dict().items()}
        unet.load_state_dict(keyed_state_dict(shapes, seed=3))
        x, ts = g(2, 4, 32, 32), torch.tensor([981.0])
        ctx, pooled, cond = g(2, 77, 2048), g(2, 1280), torch.rand(2, 3, 256, 256)
        ids = torch.tensor([[1024, 1024, 0, 0, 1024, 1024]]).repeat(2, 1)
        unet.set_timestep(ts); unet.set_clip_text_embedding(ctx); unet.set_pooled_text_embedding(pooled); unet.set_time_ids(ids)
        adapter.set_condition(cond)
        y = unet(x)
        fx.update({"cl.x": x, "cl.timestep": ts, "cl.ctx": ctx, "cl.pooled": pooled, "cl.time_ids": ids, "cl.cond": cond, "cl.y": y})
        print(f"  [ref ] SDXLUNet + ControlLora: output max {y.abs().max().item():.3f} (fixture only)")
        del unet, adapter
        out["unets"] = fx

        # ------------------------------------------------------------------------ SAM
        print("SAM ViT blocks")
        from refiners.foundationals.segment_anything.image_encoder import (
            FusedSelfAttention,
            Neck,
            PatchEncoder,
            TransformerLayer,
        )

        fx = {}
        fa = FusedSelfAttention(embedding_dim=32, spatial_size=(6, 6), num_heads=2)
        for prm in (fa.RelativePositionAttention.horizontal_embedding, fa.RelativePositionAttention.vertical_embedding):
            prm.copy_(0.3 * g(*prm.shape))
        x = g(3, 6, 6, 32)
        y = fa(x)
        fx.update({f"fsa.sd.{k}": v for k, v in fa.state_dict().items()})
        fx.update({"fsa.x": x, "fsa.y": y})
        _close("FusedSelfAttention", osam.fused_self_attention(fa.state_dict(prefix="A."), "A", x, 2), y)
        for tag, window in {"layer_win": 4, "layer_global": None}.items():
            tl = TransformerLayer(embedding_dim=32, num_heads=2, feedforward_dim=64, image_embedding_size=(10, 10), window_size=window)
            att = tl.layer(("Residual_1", "FusedSelfAttention", "RelativePositionAttention"), rfl.Module)
            for prm in (att.horizontal_embedding, att.vertical_embedding):
                prm.copy_(0.3 * g(*prm.shape))
            x = g(2, 10, 10, 32)
            y = tl(x)
            fx.update({f"{tag}.sd.{k}": v for k, v in tl.state_dict().items()})
            fx.update({f"{tag}.x": x, f"{tag}.y": y})
            _close(f"TransformerLayer window={window}", osam.transformer_layer(tl.state_dict(prefix="L."), "L", x, 2, window), y)
        pe = PatchEncoder(3, 32, patch_size=16)
        nk = Neck(in_channels=32)
        x = g(1, 3, 64, 64)
        y = pe(x)
        fx.update({f"patch.sd.{k}": v for k, v in pe.state_dict().items()})
        fx.update({"patch.x": x, "patch.y": y})
        _close("PatchEncoder", osam.patch_encoder(pe.state_dict(prefix="P."), "P", x), y)
        z = g(1, 4, 4, 32)
        yn = nk(z)
        fx.update({f"neck.sd.{k}": v for k, v in nk.state_dict().items()})
        fx.update({"neck.x": z, "neck.y": yn})
        _close("Neck", osam.neck(nk.state_dict(prefix="N."), "N", z), yn)
        out["sam"] = fx

    if write:
        GOLDEN.mkdir(parents=True, exist_ok=True)
        for name, tensors in out.items():
            path = GOLDEN / f"{name}.safetensors"
            save_file({k: v.detach().contiguous().clone() for k, v in tensors.items()}, str(path))
            print(f"wrote {path.relative_to(ROOT)} ({path.stat().st_size / 1024:.0f} KiB, {len(tensors)} tensors)")


TOKENIZER_TEXTS = [*PROMPTS, "naïve café — ünïcödé ☃ test_123 it's they're", "banana bandana " * 30, "<|startoftext|>hello<|endoftext|> world",
                   "\t tabs\nand  newlines \x7f\x80"]
LORA_SORT_KEYS = ["lora_unet_down_blocks_1_attentions_0_transformer_blocks_0_attn1_to_q", "lora_unet_down_blocks_10_attentions_0_proj_in",
                  "a_to_out_0_lora", "plain_key", "lora_te_text_model_encoder_layers_3_self_attn_k_proj", "x_in", "y_out0"]
SAM_FRAME_SIZES = ((1536, 768), (333, 517), (1024, 1024), (2000, 31))


def pin_surface(write: bool) -> None:
    """The reference's public surface, recorded for the structure and host-parity tests: repr() trees and state-dict
    contracts of every model of the hot path before / after adapter injection, and digests of the outputs of the host-side
    modules that must be bit-identical (structure.json.xz); and the CLIP merge table cut to the
    48 894 ranks the tokenizer reads (clip_merges.txt.xz)."""
    import gzip
    import json
    import lzma

    rfl = _import_reference()
    import numpy as np
    from PIL import Image

    import refiners
    import refiners.foundationals.dinov2 as rdino
    import refiners.foundationals.segment_anything.utils as rsam
    from refiners.fluxion.adapters.lora import LinearLora as RLora, LoraAdapter as RAdapter
    from refiners.fluxion.utils import gaussian_blur as rblur
    from refiners.foundationals.clip.image_encoder import CLIPImageEncoder as REnc, CLIPImageEncoderH as REncH
    from refiners.foundationals.clip.text_encoder import CLIPTextEncoderG, CLIPTextEncoderH, CLIPTextEncoderL
    from refiners.foundationals.clip.tokenizer import CLIPTokenizer
    from refiners.foundationals.latent_diffusion.auto_encoder import LatentDiffusionAutoencoder
    from refiners.foundationals.latent_diffusion.cross_attention import CrossAttentionBlock2d
    from refiners.foundationals.latent_diffusion.image_prompt import ImageProjection, IPAdapter, PerceiverResampler
    from refiners.foundationals.latent_diffusion.lora import SDLoraManager
    from refiners.foundationals.latent_diffusion.solvers import DDIM, Euler
    from refiners.foundationals.latent_diffusion.stable_diffusion_1.controlnet import SD1ControlnetAdapter
    from refiners.foundationals.latent_diffusion.stable_diffusion_1.self_attention_guidance import SD1SAGAdapter
    from refiners.foundationals.latent_diffusion.stable_diffusion_1.unet import SD1UNet
    from refiners.foundationals.latent_diffusion.stable_diffusion_xl.control_lora import ControlLoraAdapter
    from refiners.foundationals.latent_diffusion.stable_diffusion_xl.image_prompt import SDXLIPAdapter
    from refiners.foundationals.latent_diffusion.stable_diffusion_xl.self_attention_guidance import SDXLSAGAdapter
    from refiners.foundationals.latent_diffusion.stable_diffusion_xl.text_encoder import DoubleTextEncoder
    from refiners.foundationals.latent_diffusion.stable_diffusion_xl.unet import SDXLUNet
    from refiners.foundationals.latent_diffusion.style_aligned import StyleAligned
    from refiners.foundationals.segment_anything.image_encoder import SAMViTH

    from oracle.weights import keyed_state_dict
    from tests.test_lora_manager import Holder, checkpoint
    from tests.test_reference_structure import contract, digest, tree

    print("public surface: trees, contracts, host-side outputs")
    trees: dict[str, dict] = {}
    values: dict = {}

    def snap(name: str, module) -> None:
        trees[name] = {"tree": tree(module), "contract": [[k, list(s)] for k, s in contract(module)]}

    # SD 1.5 UNet + ControlNet, SDXL UNet + ControlLora + IP-Adapter
    unet = SD1UNet(4, device="meta")
    snap("sd1.unet", unet)
    adapter = SD1ControlnetAdapter(unet, name="canny", scale=0.9).inject()
    snap("sd1.unet.controlnet", unet), snap("sd1.controlnet", adapter)
    adapter.eject()
    snap("sd1.unet.controlnet_ejected", unet)
    unet = SDXLUNet(4, device="meta")
    snap("sdxl.unet", unet)
    adapter = ControlLoraAdapter("canny", unet, scale=0.8).inject()
    snap("sdxl.unet.control_lora", unet)
    adapter.eject()
    snap("sdxl.unet.control_lora_ejected", unet)
    ip = SDXLIPAdapter(unet, scale=0.5)
    ip.inject()
    snap("sdxl.unet.ip_adapter", unet), snap("sdxl.ip_adapter.image_proj", ip.image_proj)
    ip.eject()
    snap("sdxl.unet.ip_adapter_ejected", unet)

    def keyed(module, seed: int):
        module.load_state_dict(keyed_state_dict({k: tuple(v.shape) for k, v in module.state_dict().items()}, seed=seed))
        return module

    # IP-Adapter plus: the PerceiverResampler's structure and numbers (keyed weights, seeded input)
    snap("perceiver.image_proj", SDXLIPAdapter(SDXLUNet(4, device="meta"), fine_grained=True).image_proj)
    resampler = keyed(PerceiverResampler(latents_dim=64, num_attention_layers=2, num_attention_heads=4, head_dim=16, num_tokens=5, input_dim=48,
                                         output_dim=40), 31)
    with torch.no_grad():
        values["perceiver.y"] = digest(resampler(torch.randn(3, 11, 48, generator=torch.Generator().manual_seed(0))))

    # CLIP image encoder H and the IP-Adapter's image -> context path on a tiny tower
    enc_h = REncH(device="meta")
    snap("clip.image_encoder_h", enc_h), snap("clip.image_encoder_h.grid", IPAdapter.convert_to_grid_features(enc_h))
    enc = keyed(REnc(image_size=32, embedding_dim=48, output_dim=24, patch_size=8, num_layers=2, num_attention_heads=3, feedforward_dim=96), 32)
    proj = keyed(ImageProjection(clip_image_embedding_dim=24, clip_text_embedding_dim=40), 33)
    target = rfl.Chain(CrossAttentionBlock2d(channels=64, context_embedding_dim=40, context_key="ctx", num_attention_heads=2, use_linear_projection=True))
    ip = IPAdapter(target, enc, proj)
    images = torch.randn(3, 3, 32, 32, generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        values["clip.encoded"] = digest(enc(images))
        for i, kwargs in enumerate(({}, {"weights": [1.0, 0.5, 2.0]}, {"concat_batches": False})):
            values[f"clip.embedding.{i}"] = digest(ip.compute_clip_image_embedding(images, **kwargs))

    # two LoRAs on every Linear of a cross-attention block
    block = rfl.Chain(CrossAttentionBlock2d(channels=64, context_embedding_dim=48, context_key="ctx", num_attention_heads=2, num_attention_layers=2,
                                            use_linear_projection=True, device="meta"))
    snap("lora.block", block)
    for lin, parent in list(block.walk(rfl.Linear, recurse=True)):
        loras = [RLora(f"l{j}", in_features=lin.in_features, out_features=lin.out_features, rank=4, scale=s, device="meta") for j, s in enumerate((1.0, 1.4))]
        RAdapter(lin, *loras).inject(parent)
    snap("lora.block.loras", block)

    snap("sam.vit_h", SAMViTH(device="meta"))
    snap("vae", LatentDiffusionAutoencoder(device="meta"))
    for name in ("DINOv2_small", "DINOv2_base_reg", "DINOv2_large", "DINOv2_giant_reg"):
        snap(f"dinov2.{name}", getattr(rdino, name)(device="meta"))
    for tag, solver in (("euler", Euler(num_inference_steps=30)), ("ddim", DDIM(num_inference_steps=20))):
        for table in ("timesteps", "cumulative_scale_factors", "noise_std"):
            values[f"solver.{tag}.{table}"] = digest(getattr(solver, table))

    # self-attention guidance on SD 1.5 and SDXL, and the blur it uses
    for tag, unet_cls, sag_cls in (("sd1", SD1UNet, SD1SAGAdapter), ("sdxl", SDXLUNet, SDXLSAGAdapter)):
        unet = unet_cls(4, device="meta")
        sag = sag_cls(unet, scale=0.3, kernel_size=7, sigma=1.5).inject()
        snap(f"sag.{tag}.unet", unet), snap(f"sag.{tag}.adapter", sag)
        values[f"sag.{tag}.settings"] = [sag.scale, sag.kernel_size, sag.sigma]
        values[f"sag.{tag}.context_keys"] = sorted(sag.init_context().keys())
        sag.eject()
        snap(f"sag.{tag}.unet.ejected", unet)
    x = torch.randn(1, 4, 16, 20, generator=torch.Generator().manual_seed(0))
    for i, (size, sigma) in enumerate(((9, 1.0), ((3, 7), None), (5, (0.8, 2.0)))):
        values[f"sag.blur.{i}"] = digest(rblur(x, size, sigma))

    # CLIP tokenizer and text towers
    tokenizer = CLIPTokenizer()
    values["tokenizer.texts"] = TOKENIZER_TEXTS
    for i, text in enumerate(TOKENIZER_TEXTS):
        values[f"tokenizer.text.{i}"] = digest(tokenizer(text))
    values["tokenizer.batch"], values["tokenizer.encode"] = digest(tokenizer(TOKENIZER_TEXTS[:4])), digest(tokenizer.encode("hello world"))
    mapping = json.dumps(tokenizer.token_to_id_mapping, sort_keys=True, ensure_ascii=False).encode()
    values["tokenizer.mapping_sha256"] = __import__("hashlib").sha256(mapping).hexdigest()
    for cls in (CLIPTextEncoderL, CLIPTextEncoderH, CLIPTextEncoderG, DoubleTextEncoder):
        snap(f"text.{cls.__name__}", cls(device="meta"))

    # SDLoraManager on SD 1.5
    values["lora_manager.sort_keys"] = {key: list(SDLoraManager.sort_keys(key)) for key in LORA_SORT_KEYS}
    unet = SD1UNet(4, device="meta")
    manager = SDLoraManager(Holder(unet, rfl.Chain()))
    tensors = checkpoint(unet, rfl)
    values["lora_manager.checkpoint_keys"] = list(tensors)

    def lines(u) -> list[str]:  # the Lambda line prints a function signature whose annotations differ (jaxtyping): not structure
        return [line for line in repr(u).splitlines() if "Lambda(compute_sinusoidal_embedding" not in line]

    for name, scale in (("a", 0.4), ("b", 1.0)):
        manager.add_loras(name, tensors=tensors, scale=scale)
    values["lora_manager.names"], values["lora_manager.scales"] = sorted(manager.names), manager.scales
    values["lora_manager.weights_a"], values["lora_manager.tree.added"] = list(manager.get_lora_weights("a")), lines(unet)
    manager.remove_loras("a")
    values["lora_manager.tree.removed_a"] = lines(unet)
    manager.remove_all()
    values["lora_manager.tree.removed_all"] = lines(unet)

    # StyleAligned's shared-attention chain in every dtype
    for dtype in (torch.float32, torch.bfloat16, torch.float16):
        x = (torch.randn(6, 10, 16, generator=torch.Generator().manual_seed(0)) * 2 + 0.3).to(dtype)
        for i, (adain, concatenate) in enumerate(((True, False), (True, True), (False, True), (False, False))):
            values[f"style.{dtype}.{i}"] = digest(StyleAligned(adain, concatenate, 0.7)(x))

    # SAM pre- / post-processing on odd sizes
    rng, gen = np.random.default_rng(0), torch.Generator().manual_seed(0)
    for w, h in SAM_FRAME_SIZES:
        image = Image.fromarray(rng.integers(0, 255, (h, w, 3), dtype=np.uint8))
        values[f"sam.{w}x{h}.scaled_size"] = list(rsam.compute_scaled_size((h, w), 1024))
        masks, points = torch.randn(2, 3, 256, 256, generator=gen), torch.rand(2, 5, 2, generator=gen) * torch.tensor([w, h])
        values[f"sam.{w}x{h}.preprocess"] = digest(rsam.preprocess_image(image, 1024))
        values[f"sam.{w}x{h}.postprocess"] = digest(rsam.postprocess_masks(masks, (h, w), 1024))
        values[f"sam.{w}x{h}.coordinates"] = digest(rsam.normalize_coordinates(points.clone(), (h, w), 1024))

    if write:
        with lzma.open(GOLDEN / "structure.json.xz", "wt", preset=9) as f:
            json.dump({"trees": trees, "values": values}, f, ensure_ascii=False)
        with gzip.open(Path(refiners.__file__).parent / "foundationals/clip/bpe_simple_vocab_16e6.txt.gz", "rt") as f:
            merges = f.read().split("\n")[: 49152 - 256 - 2 + 1]
        with lzma.open(GOLDEN / "clip_merges.txt.xz", "wt", encoding="utf-8", preset=9 | lzma.PRESET_EXTREME) as f:
            f.write("\n".join(merges))
        for name in ("structure.json.xz", "clip_merges.txt.xz"):
            print(f"  wrote tests/golden/{name} ({(GOLDEN / name).stat().st_size / 1024:.0f} KiB)")


if __name__ == "__main__":
    write = "--check" not in sys.argv
    sections = {
        "--only-controlnet": pin_controlnet, "--only-step": pin_denoise_step, "--only-vae": pin_vae, "--only-vae-tiled": pin_vae_tiled, "--only-dinov2": pin_dinov2,
        "--only-clip": pin_clip, "--only-clip-text": pin_clip_text, "--only-sag": pin_sag, "--only-t2i": pin_t2i, "--only-style-aligned": pin_style_aligned,
        "--only-full-size": pin_full_size, "--only-surface": pin_surface,
    }
    chosen = [fn for flag, fn in sections.items() if flag in sys.argv]
    if chosen:
        for fn in chosen:
            fn(write)
    else:  # everything: the main fixture files first (one shared random stream), then the self-seeded sections
        main(write)
        for fn in sections.values():
            fn(write)

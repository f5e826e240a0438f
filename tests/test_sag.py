"""Self-attention guidance (SURVEY.md section 8f rank 4): the SAG adapters, the extra unconditional UNet pass of the
denoising step, and the attention-probability kernel behind the middle-block probe.

Fixture: tests/golden/sag.safetensors, recorded from the reference's StableDiffusion_1 with
``set_self_attention_guidance(True, scale=0.75)`` (oracle/pin_against_reference.py::pin_sag)."""

import math
from pathlib import Path

import pytest
import torch
from safetensors.torch import load_file

from oracle import sag as osag
from oracle import unet as ounet
from oracle.weights import keyed_state_dict
from refiners_b200.fluxion.utils import gaussian_blur, no_grad
from refiners_b200.foundationals.latent_diffusion import SD1UNet, SDXLUNet, StableDiffusion_1, StableDiffusion_XL
from refiners_b200.foundationals.latent_diffusion.solvers import DDIM

GOLDEN = Path(__file__).parent / "golden"
CASES = ((3, 7.5), (20, 5.0))


def keyed_unet(cls, seed, device="cpu", dtype=torch.float32):
    unet = cls(4, device="meta")
    sd = keyed_state_dict({k: tuple(v.shape) for k, v in unet.state_dict().items()}, seed=seed)
    unet.load_state_dict({k: v.to(device, dtype) for k, v in sd.items()}, assign=True)
    return unet, sd


def close(got, want, tol):
    got, want = got.float().cpu(), want.float()
    err, scale = (got - want).abs().max().item(), want.abs().max().item()
    assert err <= tol * scale, f"max abs {err:.3e} > {tol:g} x {scale:.3f}"


def test_oracle_against_the_recorded_reference():
    f = load_file(str(GOLDEN / "sag.safetensors"))
    _, sd = keyed_unet(SD1UNet, 1)
    ctx = f["sag.ctx"]
    run = lambda lat, ts, guided: ounet.sd1_unet(sd, lat, ts, ctx if guided else ctx.chunk(2)[0])  # noqa: E731
    with no_grad():
        y = osag.denoise_step(run, osag.DDIMSchedule(30), f["sag.x"], 3, 7.5, 0.75)
    close(y, f["sag.y_3"], 1e-5)


def test_sd1_step_with_sag_host():
    f = load_file(str(GOLDEN / "sag.safetensors"))
    unet, _ = keyed_unet(SD1UNet, 1)
    sd = StableDiffusion_1(unet=unet, solver=DDIM(num_inference_steps=30))
    assert not sd.has_self_attention_guidance()
    before = repr(unet)
    sd.set_self_attention_guidance(enable=True, scale=0.5)
    sd.set_self_attention_guidance(enable=True, scale=0.75)  # a second call re-scales, it does not stack adapters
    assert sd.has_self_attention_guidance() and sd._find_sag_adapter().scale == 0.75
    assert sum(type(p).__name__ == "SD1SAGAdapter" for p in unet.get_parents()) == 1
    with no_grad():
        for step, scale in CASES:
            close(sd(f["sag.x"], step=step, clip_text_embedding=f["sag.ctx"], condition_scale=scale), f[f"sag.y_{step}"], 1e-5)
    sd.set_self_attention_guidance(enable=False)
    assert not sd.has_self_attention_guidance() and repr(unet) == before and unet.parent is None


def test_gaussian_blur_is_a_normalised_reflecting_filter():
    x = torch.randn(2, 3, 12, 10)
    assert torch.allclose(gaussian_blur(torch.ones(1, 2, 9, 9), 5, 1.3), torch.ones(1, 2, 9, 9), atol=1e-6)
    assert gaussian_blur(x, (3, 5)).shape == x.shape  # default sigma, (kx, ky) sizes
    assert torch.allclose(gaussian_blur(x, 9, 1.0), osag.gaussian_blur(x, 9, 1.0), atol=1e-6)


def test_structure_against_the_reference():
    """Trees with the probes in place, the adapter's own tree, and what eject leaves behind - SD 1.5 and SDXL - against the
    reference's recording (tests/golden/structure.json.xz)."""
    from tests.test_reference_structure import digest, recorded_values, same, same_tree

    from refiners_b200.foundationals.latent_diffusion.stable_diffusion_1.self_attention_guidance import SD1SAGAdapter
    from refiners_b200.foundationals.latent_diffusion.stable_diffusion_xl.self_attention_guidance import SDXLSAGAdapter

    for tag, mine_cls, mine_ad in (("sd1", SD1UNet, SD1SAGAdapter), ("sdxl", SDXLUNet, SDXLSAGAdapter)):
        mine = mine_cls(4, device="meta")
        a = mine_ad(mine, scale=0.3, kernel_size=7, sigma=1.5).inject()
        same(mine, f"sag.{tag}.unet")
        same_tree(a, f"sag.{tag}.adapter")
        assert [a.scale, a.kernel_size, a.sigma] == recorded_values(f"sag.{tag}.settings")
        assert sorted(a.init_context().keys()) == recorded_values(f"sag.{tag}.context_keys")
        a.eject()
        same(mine, f"sag.{tag}.unet.ejected")
    x = torch.randn(1, 4, 16, 20, generator=torch.Generator().manual_seed(0))
    for i, (size, sigma) in enumerate(((9, 1.0), ((3, 7), None), (5, (0.8, 2.0)))):
        assert digest(gaussian_blur(x, size, sigma)) == recorded_values(f"sag.blur.{i}")


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("shape", [(2, 8, 64, 64, 40), (1, 20, 1024, 1024, 64), (3, 2, 50, 77, 16), (1, 1, 5, 3000, 256)])
def test_attention_probs_kernel(dtype, shape):
    """rb200_attention_probs against softmax(q k^T / sqrt(d)) in fp32 from the same (rounded) operands: one rounding
    of the stored probability."""
    from refiners_b200 import backend as B

    batch, heads, sq, sk, d = shape
    gen = torch.Generator().manual_seed(sum(shape))
    q = torch.randn(batch, sq, heads * d, generator=gen).to("cuda", dtype)
    k = torch.randn(batch, sk, heads * d, generator=gen).to("cuda", dtype)
    got = B.attention_probs(q, k, heads)
    split = lambda t, s: t.float().reshape(batch, s, heads, d).transpose(1, 2)  # noqa: E731
    want = torch.softmax(split(q, sq) @ split(k, sk).transpose(-1, -2) / math.sqrt(d), dim=-1)
    assert got.shape == want.shape and got.dtype == dtype
    eps = {torch.float32: 2e-6, torch.bfloat16: 2**-8, torch.float16: 2**-11}[dtype]
    assert (got.float() - want).abs().max().item() <= eps * max(want.max().item(), 1e-3) + 1e-7
    assert (got.float().sum(-1) - 1).abs().max().item() <= (4 * eps if dtype != torch.float32 else 1e-5)
    # strided views (the q / k slices of a fused projection) are read in place
    qkv = torch.randn(batch, sq, 3 * heads * d, generator=gen).to("cuda", dtype)
    qs, ks = qkv[..., : heads * d], qkv[..., heads * d : 2 * heads * d]
    assert torch.equal(B.attention_probs(qs, ks, heads), B.attention_probs(qs.contiguous(), ks.contiguous(), heads))


@pytest.mark.gpu
def test_sd1_step_with_sag_gpu():
    """The recorded reference step through the CUDA path in fp32 (the mask is a threshold: only fp32 is compared value
    by value), eager and with the CUDA graph switched on (a guided model keeps running the walker)."""
    f = load_file(str(GOLDEN / "sag.safetensors"))
    unet, _ = keyed_unet(SD1UNet, 1, "cuda")
    sd = StableDiffusion_1(unet=unet, solver=DDIM(num_inference_steps=30, device="cuda"), device="cuda")
    sd.set_self_attention_guidance(enable=True, scale=0.75)
    x, ctx = f["sag.x"].cuda(), f["sag.ctx"].cuda()
    with no_grad():
        for step, scale in CASES:
            close(sd(x, step=step, clip_text_embedding=ctx, condition_scale=scale), f[f"sag.y_{step}"], 2e-4)
        sd.enable_cuda_graph()
        for _ in range(4):  # more steps than the capture warm-up would have pushed shapes for
            y = sd(x, step=3, clip_text_embedding=ctx, condition_scale=7.5)
        close(y, f["sag.y_3"], 2e-4)


@pytest.mark.gpu
def test_sdxl_step_with_sag_gpu():
    """SDXL (first of the middle block's ten self-attentions is probed; pooled embedding and time ids are halved for
    the extra pass) against the oracle on the same keyed weights, fp32, 32x32 latents."""
    unet, sd_cpu = keyed_unet(SDXLUNet, 2, "cuda")
    gen = torch.Generator().manual_seed(99)
    x, ctx = torch.randn(1, 4, 32, 32, generator=gen), torch.randn(2, 77, 2048, generator=gen)
    pooled, ids = torch.randn(2, 1280, generator=gen), torch.tensor([[1024.0, 1024, 0, 0, 1024, 1024]] * 2)
    sdxl = StableDiffusion_XL(unet=unet, solver=DDIM(num_inference_steps=30, device="cuda"), device="cuda")
    sdxl.set_self_attention_guidance(enable=True, scale=1.0)

    def run(lat, ts, guided):
        half = slice(None) if guided else slice(0, 1)
        return ounet.sdxl_unet(sd_cpu, lat, ts, ctx[half], pooled[half], ids[half])

    with no_grad():
        want = osag.denoise_step(run, osag.DDIMSchedule(30), x, 10, 5.0, 1.0)
        got = sdxl(x.cuda(), step=10, clip_text_embedding=ctx.cuda(), pooled_text_embedding=pooled.cuda(), time_ids=ids.cuda(),
                   condition_scale=5.0)
    close(got, want, 2e-4)

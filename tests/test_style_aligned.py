"""StyleAligned shared attention (SURVEY.md section 8f rank 4) against tests/golden/style_aligned.safetensors, recorded from the
reference with the adapter on SD1UNet / SDXLUNet (oracle/pin_against_reference.py --only-style-aligned)."""

from pathlib import Path

import pytest
import torch
from safetensors.torch import load_file

from oracle.cases import keyed_input
from oracle.weights import keyed_state_dict
from refiners_b200.fluxion.utils import no_grad
from refiners_b200.foundationals.latent_diffusion import SD1UNet, SDXLUNet
from refiners_b200.foundationals.latent_diffusion.style_aligned import StyleAligned, StyleAlignedAdapter

GOLDEN = Path(__file__).parent / "golden"
CASES = {"sd1": (SD1UNet, 1, 768), "sdxl": (SDXLUNet, 2, 2048)}


def run(tag, device, dtype):
    unet_cls, seed, width = CASES[tag]
    unet = unet_cls(4, device="meta")
    sd = keyed_state_dict({k: tuple(v.shape) for k, v in unet.state_dict().items()}, seed=seed)
    unet.load_state_dict({k: v.to(device, dtype) for k, v in sd.items()}, assign=True)
    adapter = StyleAlignedAdapter(unet, scale=0.7).inject()
    unet.set_timestep(torch.tensor([601.0], device=device))
    unet.set_clip_text_embedding(keyed_input(f"style.{tag}.ctx", (4, 77, width)).to(device, dtype))
    if tag == "sdxl":
        unet.set_pooled_text_embedding(keyed_input("style.sdxl.pooled", (4, 1280)).to(device, dtype))
        unet.set_time_ids(torch.tensor([[1024.0, 1024, 0, 0, 1024, 1024]] * 4, device=device))
    with no_grad():
        y = unet(keyed_input(f"style.{tag}.x", (4, 4, 32, 32)).to(device, dtype))
    adapter.eject()
    return y


def close(got, want, tol):
    got, want = got.float().cpu(), want.float()
    err, scale = (got - want).abs().max().item(), want.abs().max().item()
    assert err <= tol * scale, f"max abs {err:.3e} > {tol:g} x {scale:.3f}"


@pytest.mark.parametrize("tag", ["sd1", "sdxl"])
def test_style_aligned_host(tag):
    close(run(tag, "cpu", torch.float32), load_file(str(GOLDEN / "style_aligned.safetensors"))[f"{tag}.y"], 1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=str)
@pytest.mark.parametrize("tag", ["sd1", "sdxl"])
def test_style_aligned_gpu(cuda_device, tag, dtype):
    close(run(tag, cuda_device, dtype), load_file(str(GOLDEN / "style_aligned.safetensors"))[f"{tag}.y"], 2e-4 if dtype == torch.float32 else 5e-2)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16], ids=str)
@pytest.mark.parametrize("variant", [(True, False), (True, True), (False, True), (False, False)], ids=["q", "k", "v", "plain"])
def test_style_aligned_kernel(cuda_device, variant, dtype):
    """rb200_style_aligned against the module-by-module evaluation in fp32 on the same (rounded) input, contiguous and as a
    strided slice of a fused projection; the fused path and the generic path of the chain agree."""
    adain, concatenate = variant
    gen = torch.Generator().manual_seed(3)
    packed = (torch.randn(6, 50, 3 * 40, generator=gen) * 1.5 + 0.3).to(cuda_device, dtype)
    x = packed[..., 40:80]
    chain = StyleAligned(adain=adain, concatenate=concatenate, scale=0.6)
    with no_grad():
        got = chain(x)
        want = chain(x.float().cpu())
        chain.register_forward_hook(lambda *_: None)  # a hooked chain takes the generic path
        generic = chain(x.contiguous())
    assert got.shape == want.shape and got.dtype == dtype
    eps = {torch.float32: 2e-6, torch.bfloat16: 2**-8, torch.float16: 2**-11}[dtype]
    assert (got.float().cpu() - want).abs().max().item() <= eps * want.abs().max().item()
    assert (generic.float() - got.float()).abs().max().item() <= 8 * eps * want.abs().max().item()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16], ids=str)
def test_style_aligned_chain_is_bit_identical_to_the_reference_on_the_host(dtype):
    from tests.test_reference_structure import digest, recorded_values

    x = (torch.randn(6, 10, 16, generator=torch.Generator().manual_seed(0)) * 2 + 0.3).to(dtype)
    for i, (adain, concatenate) in enumerate(((True, False), (True, True), (False, True), (False, False))):
        assert digest(StyleAligned(adain, concatenate, 0.7)(x)) == recorded_values(f"style.{dtype}.{i}"), (adain, concatenate)

"""SAM ViT blocks and IP-Adapter / LoRA injection against golden vectors and the oracle.

Host tests: fp32 on CPU (<= 1e-5 relative).  GPU tests: the same graphs through the C-ABI
kernels, fused vs unfused execution, fp32 2e-4 / 16-bit 5 % max-abs + 1 % mean-abs of max|ref|."""

from pathlib import Path

import pytest
import torch
from safetensors.torch import load_file

import refiners_b200.fluxion.layers as fl
from oracle import ops as oops
from refiners_b200.fluxion.adapters import LinearLora, LoraAdapter, auto_attach_loras
from refiners_b200.fluxion.utils import no_grad
from refiners_b200.foundationals.latent_diffusion import CrossAttentionBlock2d
from refiners_b200.foundationals.latent_diffusion.image_prompt import CrossAttentionAdapter, ImageCrossAttention, SDXLIPAdapter
from refiners_b200.foundationals.segment_anything.image_encoder import FusedSelfAttention, Neck, PatchEncoder, TransformerLayer
from tests.test_models_golden import check, sub

GOLDEN = Path(__file__).parent / "golden"


@pytest.fixture(scope="module")
def sam():
    return load_file(str(GOLDEN / "sam.safetensors"))


def sam_cases(sam):
    fa = FusedSelfAttention(embedding_dim=32, spatial_size=(6, 6), num_heads=2)
    fa.load_state_dict(sub(sam, "fsa.sd."))
    yield "fsa", fa
    for tag, window in (("layer_win", 4), ("layer_global", None)):
        tl = TransformerLayer(embedding_dim=32, num_heads=2, feedforward_dim=64, image_embedding_size=(10, 10), window_size=window)
        tl.load_state_dict(sub(sam, f"{tag}.sd."))
        yield tag, tl
    pe = PatchEncoder(3, 32, patch_size=16)
    pe.load_state_dict(sub(sam, "patch.sd."))
    yield "patch", pe
    nk = Neck(in_channels=32)
    nk.load_state_dict(sub(sam, "neck.sd."))
    yield "neck", nk


def test_sam_blocks_host(sam):
    with no_grad():
        for tag, module in sam_cases(sam):
            check(module(sam[f"{tag}.x"]), sam[f"{tag}.y"], "host")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=str)
def test_sam_blocks_gpu(cuda_device, sam, dtype):
    with no_grad():
        for tag, module in sam_cases(sam):
            y = module.to(cuda_device, dtype)(sam[f"{tag}.x"].to(cuda_device, dtype))
            check(y, sam[f"{tag}.y"], dtype)


def make_ip_block(seed=0):
    torch.manual_seed(seed)
    ca = CrossAttentionBlock2d(64, context_embedding_dim=48, context_key="ctx", num_attention_heads=1, num_attention_layers=1,
                               use_bias=False, use_linear_projection=True)
    top = fl.Chain(ca)
    adapters = [CrossAttentionAdapter(target=a, scale=0.7) for a in ca.layers(fl.Attention, recurse=True) if type(a) is not fl.SelfAttention]
    assert len(adapters) == 1
    return top, ca, adapters


def ip_reference(ca, adapter, x, ctx, img):
    """Oracle-style evaluation: out = SDPA(q, k_t, v_t) + s * SDPA(q, Wk' e, Wv' e) inside the block."""
    from oracle import unet as ounet

    sd = {"X." + k: v for k, v in ca.state_dict().items()}
    # strip the adapter from the keys to obtain the plain block, then patch the attention by hand
    attn_prefix = next(k for k in sd if "Residual_2" in k and "Distribute.Linear_1.weight" in k).rsplit(".Distribute", 1)[0]
    plain = {k.replace(".CrossAttentionAdapter.Attention", ".Attention").replace(".Sum.ImageCrossAttention", ".IMG"): v for k, v in sd.items()}
    B_, C, H, W = x.shape
    c1 = "X.Chain_1"
    h = oops.group_norm(x, 32, plain[c1 + ".GroupNorm.weight"], plain[c1 + ".GroupNorm.bias"], 1e-6)
    h = oops.linear(h.flatten(2).transpose(1, 2), plain[c1 + ".Linear.weight"], plain[c1 + ".Linear.bias"])
    blk = "X.Chain_2.CrossAttentionBlock"
    r1, r2, r3 = blk + ".Residual_1", blk + ".Residual_2", blk + ".Residual_3"
    n = oops.layer_norm(h, plain[r1 + ".LayerNorm.weight"], plain[r1 + ".LayerNorm.bias"], 1e-5)
    h = h + ounet.attention(plain, r1 + ".SelfAttention", n, n, 1)
    n = oops.layer_norm(h, plain[r2 + ".LayerNorm.weight"], plain[r2 + ".LayerNorm.bias"], 1e-5)
    a = r2 + ".Attention"
    q = oops.linear(n, plain[a + ".Distribute.Linear_1.weight"])
    kt, vt = oops.linear(ctx, plain[a + ".Distribute.Linear_2.weight"]), oops.linear(ctx, plain[a + ".Distribute.Linear_3.weight"])
    ki = oops.linear(img, plain[a + ".IMG.Distribute.Chain_1.Linear.weight"])
    vi = oops.linear(img, plain[a + ".IMG.Distribute.Chain_2.Linear.weight"])
    o = oops.sdpa(q, kt, vt, 1) + adapter.scale * oops.sdpa(q, ki, vi, 1)
    h = h + oops.linear(o, plain[a + ".Linear.weight"], plain[a + ".Linear.bias"])
    n = oops.layer_norm(h, plain[r3 + ".LayerNorm.weight"], plain[r3 + ".LayerNorm.bias"], 1e-5)
    h = h + oops.linear(oops.glu_gelu(oops.linear(n, plain[r3 + ".Linear_1.weight"], plain[r3 + ".Linear_1.bias"])), plain[r3 + ".Linear_2.weight"], plain[r3 + ".Linear_2.bias"])
    h = oops.linear(h, plain["X.Chain_3.Linear.weight"], plain["X.Chain_3.Linear.bias"]).transpose(1, 2).reshape(B_, C, H, W)
    del attn_prefix
    return h + x


def run_ip(top, ca, adapters, device, dtype, x, ctx, img):
    top = top.to(device, dtype)
    for ad in adapters:
        ad.image_cross_attention.to(device, dtype)
    top.set_context("cross_attention_block", {"ctx": ctx.to(device, dtype)})
    top.set_context("ip_adapter", {"clip_image_embedding": img.to(device, dtype)})
    with no_grad():
        return top(x.to(device, dtype))


def test_ip_adapter_inject_eject_and_formula_host():
    top, ca, adapters = make_ip_block()
    before = repr(top)
    n_keys = len(top.state_dict())
    for ad in adapters:
        ad.inject()
    assert len(top.state_dict()) == n_keys + 2
    assert any(".Sum.ImageCrossAttention.Distribute.Chain_1.Linear.weight" in k for k in top.state_dict())
    g = torch.Generator().manual_seed(5)
    x, ctx, img = torch.randn(2, 64, 4, 4, generator=g), torch.randn(2, 5, 48, generator=g), torch.randn(2, 4, 48, generator=g)
    y = run_ip(top, ca, adapters, "cpu", torch.float32, x, ctx, img)
    check(y, ip_reference(ca, adapters[0], x, ctx, img), "host")
    for ad in adapters:
        ad.eject()
    assert repr(top) == before and len(top.state_dict()) == n_keys


def test_sdxl_ip_adapter_structure():
    from refiners_b200.foundationals.latent_diffusion import SDXLUNet

    unet = SDXLUNet(4, device="meta")
    before = repr(unet)
    ip = SDXLIPAdapter(unet, scale=0.5)
    assert len(ip.sub_adapters) == 70          # every non-self attention of SDXL
    ip.inject()
    assert unet.parent is ip and len(list(unet.layers(ImageCrossAttention, recurse=True))) == 70
    ip.scale = 0.25
    assert all(s.scale == 0.25 for s in ip.sub_adapters)
    ip.eject()
    assert repr(unet) == before and unet.parent is None


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=str)
@pytest.mark.parametrize("fusion", [True, False], ids=["fused", "unfused"])
def test_ip_adapter_gpu(cuda_device, dtype, fusion):
    from refiners_b200 import backend as B

    top, ca, adapters = make_ip_block()
    for ad in adapters:
        ad.inject()
    g = torch.Generator().manual_seed(5)
    x, ctx, img = torch.randn(2, 64, 8, 8, generator=g), torch.randn(2, 5, 48, generator=g), torch.randn(2, 4, 48, generator=g)
    ref = ip_reference(ca, adapters[0], x, ctx, img)
    prev = B.set_fusion(fusion)
    try:
        check(run_ip(top, ca, adapters, cuda_device, dtype, x, ctx, img), ref, dtype)
    finally:
        B.set_fusion(prev)


def make_lora_block(oracle_loras: dict | None = None):
    """``oracle_loras`` (optional) receives {original path of the adapted Linear: [(down, up, scale), ...]} - the
    description oracle.unet.Weights wants."""
    torch.manual_seed(3)
    ca = CrossAttentionBlock2d(64, context_embedding_dim=48, context_key="ctx", num_attention_heads=1, num_attention_layers=1,
                               use_bias=False, use_linear_projection=True)
    top = fl.Chain(ca)
    plain_sd = {k: v.clone() for k, v in top.state_dict().items()}
    paths = {id(m): name for name, m in top.named_modules()}
    targets = [(m, p) for m, p in top.walk(fl.Linear, recurse=True) if "CrossAttentionBlock" in {type(a).__name__ for a in p.get_parents() + [p]}]
    for i, (lin, parent) in enumerate(targets):
        loras = []
        for j, (rank, scale) in enumerate(((4, 1.0), (8, 1.4))):
            lora = LinearLora(f"l{j}", in_features=lin.in_features, out_features=lin.out_features, rank=rank, scale=scale)
            lora.up.weight.data.normal_(0, 0.05)
            loras.append(lora)
            if oracle_loras is not None:
                oracle_loras.setdefault(paths[id(lin)], []).append((lora.down.weight.detach().clone(), lora.up.weight.detach().clone(), scale))
        LoraAdapter(lin, *loras).inject(parent)
    return top, ca, plain_sd


def test_lora_injection_matches_merged_weights_host():
    """700-adapter style injection on a small block: y(adapted) == y(plain block with W + sum s B A)."""
    top, ca, plain_sd = make_lora_block()
    adapters = list(top.layers(LoraAdapter, recurse=True))
    assert len(adapters) == 10  # q,k,v,o x2 + 2 MLP linears of the block
    g = torch.Generator().manual_seed(6)
    x, ctx = torch.randn(2, 64, 4, 4, generator=g), torch.randn(2, 5, 48, generator=g)
    top.set_context("cross_attention_block", {"ctx": ctx})
    with no_grad():
        y = top(x)
    merged = CrossAttentionBlock2d(64, context_embedding_dim=48, context_key="ctx", num_attention_heads=1, num_attention_layers=1,
                                   use_bias=False, use_linear_projection=True)
    merged_top = fl.Chain(merged)
    merged_top.load_state_dict(plain_sd)
    plain_linears = [m for m, p in merged_top.walk(fl.Linear, recurse=True)
                     if "CrossAttentionBlock" in {type(a).__name__ for a in p.get_parents() + [p]}]
    assert len(plain_linears) == len(adapters)
    for lin, ad in zip(plain_linears, adapters):  # same depth-first order in both trees
        delta = sum(l.scale * (l.up.weight @ l.down.weight) for l in ad.lora_layers)
        lin.weight.data = ad.target.weight.data + delta
    merged_top.set_context("cross_attention_block", {"ctx": ctx})
    with no_grad():
        check(y, merged_top(x), "host")


def test_lora_block_oracle_host():
    """The host mirror of a LoRA-adapted block against the ORACLE restatement (oracle.unet with Weights.loras)."""
    from oracle import unet as ounet

    desc: dict = {}
    top, ca, plain_sd = make_lora_block(desc)
    g = torch.Generator().manual_seed(6)
    x, ctx = torch.randn(2, 64, 8, 8, generator=g), torch.randn(2, 5, 48, generator=g)
    top.set_context("cross_attention_block", {"ctx": ctx})
    with no_grad():
        y = top(x)
        ref = ounet.cross_attention_2d(ounet.Weights(plain_sd, loras=desc), "CrossAttentionBlock2d", x, ctx, 1, 1, True)
    check(y, ref, "host")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=str)
@pytest.mark.parametrize("fusion", ["merged", "two-launch", "unfused"])
def test_lora_block_gpu(cuda_device, dtype, fusion):
    """A LoRA-adapted CrossAttentionBlock2d (10 adapters, 2 LoRAs each) on the kernels against the oracle restatement
    evaluated in fp32 on the CPU: with the merged-weight evaluation (default), the two-launch evaluation and unfused."""
    from oracle import unet as ounet
    from refiners_b200 import backend as B

    desc: dict = {}
    top, ca, plain_sd = make_lora_block(desc)
    g = torch.Generator().manual_seed(6)
    x, ctx = torch.randn(2, 64, 8, 8, generator=g), torch.randn(2, 5, 48, generator=g)
    with no_grad():
        ref = ounet.cross_attention_2d(ounet.Weights(plain_sd, loras=desc), "CrossAttentionBlock2d", x, ctx, 1, 1, True)
    prev = B.set_fusion(fusion != "unfused")
    prev_merge = B.set_lora_merge(fusion == "merged")
    try:
        top = top.to(cuda_device, dtype)
        top.set_context("cross_attention_block", {"ctx": ctx.to(cuda_device, dtype)})
        before = B.launch_count()
        with no_grad():
            y = top(x.to(cuda_device, dtype))
        launches = B.launch_count() - before
        check(y, ref, dtype)
    finally:
        B.set_fusion(prev)
        B.set_lora_merge(prev_merge)
    assert launches > 0


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=str)
@pytest.mark.parametrize("stride", [1, 2])
def test_conv2d_lora_gpu(cuda_device, dtype, stride):
    """LoraAdapter around a Conv2d with a Conv2dLora (1x1 down with the target's stride, 3x3 up; lora.py:269-380 of the
    reference): every conv of the Sum runs on the kernels; checked against y = conv(x) + s * up(down(x)) in fp32."""
    import torch.nn.functional as F

    from refiners_b200 import backend as B
    from refiners_b200.fluxion.adapters import Conv2dLora

    torch.manual_seed(11)
    conv = fl.Conv2d(64, 96, kernel_size=3, stride=stride, padding=1)
    holder = fl.Chain(conv)
    lora = Conv2dLora("c", in_channels=64, out_channels=96, rank=8, scale=1.3)
    lora.up.weight.data.normal_(0, 0.05)
    adapter = LoraAdapter(conv, lora)
    assert lora.is_compatible(conv) and tuple(lora.down.stride) == (stride, stride)
    adapter.inject(holder)
    x = torch.randn(2, 64, 16, 16)
    rd = lambda t: t.detach().to(dtype).float()  # what the kernels see
    ref = F.conv2d(rd(x), rd(conv.weight), rd(conv.bias), stride=stride, padding=1) + 1.3 * F.conv2d(
        F.conv2d(rd(x), rd(lora.down.weight), None, stride=stride), rd(lora.up.weight), None, padding=1)
    holder = holder.to(cuda_device, dtype)
    before = B.launch_count()
    with no_grad():
        y = holder(x.to(cuda_device, dtype))
    assert B.launch_count() - before >= 3  # base conv, down, up (+ scale / add)
    check(y, ref, dtype)


def test_sam_image_frame_matches_the_reference():
    """Pre- / post-processing around the encoder (segment_anything/utils.py:7-130): bit-identical to the reference's
    recording on odd sizes."""
    import numpy as np
    from PIL import Image

    import refiners_b200.foundationals.segment_anything.utils as mine
    from tests.test_reference_structure import digest, recorded_values

    rng, gen = np.random.default_rng(0), torch.Generator().manual_seed(0)
    for w, h in ((1536, 768), (333, 517), (1024, 1024), (2000, 31)):
        image = Image.fromarray(rng.integers(0, 255, (h, w, 3), dtype=np.uint8))
        assert list(mine.compute_scaled_size((h, w), 1024)) == recorded_values(f"sam.{w}x{h}.scaled_size")
        masks, points = torch.randn(2, 3, 256, 256, generator=gen), torch.rand(2, 5, 2, generator=gen) * torch.tensor([w, h])
        assert digest(mine.preprocess_image(image, 1024)) == recorded_values(f"sam.{w}x{h}.preprocess"), (w, h)
        assert digest(mine.postprocess_masks(masks, (h, w), 1024)) == recorded_values(f"sam.{w}x{h}.postprocess"), (w, h)
        assert digest(mine.normalize_coordinates(points.clone(), (h, w), 1024)) == recorded_values(f"sam.{w}x{h}.coordinates"), (w, h)

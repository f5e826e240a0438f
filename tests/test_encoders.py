"""DINOv2 and CLIP vision towers (SURVEY.md section 8f rank 3) against reference-recorded fixtures
(tests/golden/dinov2.safetensors, clip.safetensors; oracle/pin_against_reference.py --only-dinov2 / --only-clip):
host path (fp32, <= 1e-5 relative) and the same graphs on the CUDA kernels - fp32 within 2e-4 relative, bf16 under the
criterion of tests/test_full_size_gpu.py (error vs the reference's fp32 output no larger than that of torch-eager bf16 on
the same GPU + 1e-3 max|ref|)."""

import gzip
import hashlib
import json
import lzma
from pathlib import Path

import pytest
import torch
from safetensors.torch import load_file

import refiners_b200.fluxion.layers as fl
from oracle import clip as oclip
from oracle import dinov2 as odino
from oracle import ops as oops
from oracle.cases import keyed_input
from oracle.weights import keyed_state_dict
from refiners_b200.fluxion.utils import no_grad

GOLDEN = Path(__file__).parent / "golden"


def keyed(model, seed, device="cpu", dtype=torch.float32):
    sd = keyed_state_dict({k: tuple(v.shape) for k, v in model.state_dict().items()}, seed=seed)
    model.load_state_dict({k: v.to(device, dtype) for k, v in sd.items()}, assign=True)
    return model


def rel_err(got, want):
    got, want = got.float().cpu(), want.float().cpu()
    scale = max(want.abs().max().item(), 1e-3)
    d = got - want
    return d.abs().max().item() / scale, d.pow(2).mean().sqrt().item() / scale


def build(case: str, device="cpu", dtype=torch.float32):
    """(model, input, oracle evaluation on a state dict, fixture key)"""
    if case == "clip_h":
        from refiners_b200.foundationals.clip import CLIPImageEncoderH

        return (keyed(CLIPImageEncoderH(device="meta"), 9, device, dtype), keyed_input("clip.h.image", (2, 3, 224, 224)),
                lambda sd, x: oclip.image_encoder(sd, x, patch_size=14, num_layers=32, num_heads=16), ("clip", "h.y"))
    if case == "clip_tiny":
        from refiners_b200.foundationals.clip import CLIPImageEncoder

        m = CLIPImageEncoder(image_size=32, embedding_dim=32, output_dim=16, patch_size=8, num_layers=2, num_attention_heads=2,
                             feedforward_dim=64, device="meta")
        return (keyed(m, 10, device, dtype), keyed_input("clip.tiny.image", (3, 3, 32, 32)),
                lambda sd, x: oclip.image_encoder(sd, x, patch_size=8, num_layers=2, num_heads=2), ("clip", "tiny.y"))
    if case == "dinov2_small":
        from refiners_b200.foundationals.dinov2 import DINOv2_small

        return (keyed(DINOv2_small(device="meta"), 6, device, dtype), None,
                lambda sd, x: odino.vit(sd, x, patch_size=14, num_layers=12, num_heads=6), ("dinov2", "small"))
    if case == "dinov2_tiny":
        from refiners_b200.foundationals.dinov2 import ViT

        m = ViT(embedding_dim=64, patch_size=4, image_size=16, num_layers=2, num_heads=2, num_registers=3, feedforward_dim=96,
                interpolate_antialias=True, activation=fl.GLU(fl.SiLU()), device="meta")
        return (keyed(m, 7, device, dtype), None,
                lambda sd, x: odino.vit(sd, x, patch_size=4, num_layers=2, num_heads=2, num_registers=3, swiglu=True, interpolate_antialias=True),
                ("dinov2", "tiny"))
    raise KeyError(case)


def fixture(case_key, x):
    file, key = case_key
    f = load_file(str(GOLDEN / f"{file}.safetensors"))
    if file == "dinov2":
        return f[f"{key}.x"], f[f"{key}.y"]
    return x, f[key]


@pytest.mark.parametrize("case", ["clip_tiny", "clip_h"])
def test_clip_image_encoder_host(case):
    model, x, _, key = build(case)
    x, want = fixture(key, x)
    with no_grad():
        e_max, _ = rel_err(model(x), want)
    assert e_max <= 2e-5, f"{case}: {e_max:.3e}"


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=str)
@pytest.mark.parametrize("case", ["clip_tiny", "clip_h", "dinov2_tiny", "dinov2_small"])
def test_vision_tower_gpu(cuda_device, case, dtype):
    from refiners_b200 import backend as B

    model, x, oracle_eval, key = build(case, cuda_device, dtype)
    x, want = fixture(key, x)
    xd = x.to(cuda_device, dtype)
    before = B.launch_count()
    with no_grad():
        y = model(xd)
        assert torch.equal(y, model(xd)), "two identical forwards must be bit-identical"
    assert B.launch_count() > before
    e_max, e_rms = rel_err(y, want)
    if dtype == torch.float32:
        print(f"\n[{case} fp32] max-abs {e_max:.3e} of max|ref|")
        assert e_max <= 2e-4
        return
    prev, oops.FAST = oops.FAST, True
    try:
        with torch.no_grad():
            eager = oracle_eval(dict(model.state_dict()), xd)
    finally:
        oops.FAST = prev
    t_max, t_rms = rel_err(eager, want)
    print(f"\n[{case} bf16] engine max-abs {e_max:.3e} rms {e_rms:.3e} | torch-eager bf16 max-abs {t_max:.3e} rms {t_rms:.3e} (relative to max|ref|)")
    assert e_rms <= t_rms + 1e-3 and e_max <= 1.25 * t_max + 1e-3


# ------------------------------------------------------------------------------------------ CLIP text towers
PROMPTS = ["a photo of a cat", "", "An astronaut riding a horse on Mars, 4k, highly-detailed!!"]


def text_tower(device="cpu", dtype=torch.float32):
    from refiners_b200.foundationals.clip import CLIPTextEncoderL

    return keyed(CLIPTextEncoderL(device="meta"), 21, device, dtype)


def double_tower(device, dtype):
    from refiners_b200.foundationals.latent_diffusion.stable_diffusion_xl.text_encoder import DoubleTextEncoder

    return keyed(DoubleTextEncoder(device="meta"), 22, device, dtype)


def test_clip_text_encoder_host():
    """CLIPTextEncoderL on recorded token ids (no vocabulary file needed) against the reference's output; the oracle too."""
    f = load_file(str(GOLDEN / "clip_text.safetensors"))
    tower = text_tower()
    with no_grad():
        e_max, _ = rel_err(tower(f["l.tokens"]), f["l.y"])
        o_max, _ = rel_err(oclip.text_encoder(dict(tower.state_dict()), f["l.tokens"], num_layers=12, heads=12, quick_gelu=True), f["l.y"])
    assert e_max <= 1e-5 and o_max <= 1e-5, (e_max, o_max)


@pytest.fixture(scope="module")
def vocabulary(tmp_path_factory) -> Path:
    """The CLIP merge table (data published with OpenAI CLIP), cut to the ranks the tokenizer reads and stored as xz; the
    tokenizer reads it gzipped, as it is published."""
    path = tmp_path_factory.mktemp("clip") / "bpe_simple_vocab_16e6.txt.gz"
    with lzma.open(GOLDEN / "clip_merges.txt.xz", "rb") as src, gzip.open(path, "wb") as dst:
        dst.write(src.read())
    return path


def test_clip_tokenizer_against_the_reference(vocabulary):
    """Token ids, the token -> id table and the text towers' structure against the reference's recording."""
    from refiners_b200.foundationals.clip import CLIPTokenizer
    from tests.test_reference_structure import digest, recorded_values, same

    mine = CLIPTokenizer(vocabulary_path=vocabulary)
    f = load_file(str(GOLDEN / "clip_text.safetensors"))
    assert torch.equal(mine(PROMPTS), f["l.tokens"]) and torch.equal(CLIPTokenizer(vocabulary_path=vocabulary, pad_token_id=0)(PROMPTS), f["xl.tokens_g"])
    texts = recorded_values("tokenizer.texts")
    for i, text in enumerate(texts):
        assert digest(mine(text)) == recorded_values(f"tokenizer.text.{i}"), text
    assert digest(mine(texts[:4])) == recorded_values("tokenizer.batch") and digest(mine.encode("hello world")) == recorded_values("tokenizer.encode")
    mapping = json.dumps(mine.token_to_id_mapping, sort_keys=True, ensure_ascii=False).encode()
    assert hashlib.sha256(mapping).hexdigest() == recorded_values("tokenizer.mapping_sha256")
    # trees and state-dict contract of the towers and of SDXL's double encoder (pooling adapter injected)
    from refiners_b200.foundationals.clip import CLIPTextEncoderG, CLIPTextEncoderH, CLIPTextEncoderL
    from refiners_b200.foundationals.latent_diffusion.stable_diffusion_xl.text_encoder import DoubleTextEncoder

    for ours in (CLIPTextEncoderL, CLIPTextEncoderH, CLIPTextEncoderG, DoubleTextEncoder):
        same(ours(device="meta"), f"text.{ours.__name__}")
    twin = DoubleTextEncoder(device="meta").structural_copy()
    same(twin, "text.DoubleTextEncoder")


def test_prompt_embedding_api():
    """LatentDiffusionModel.compute_clip_text_embedding: (negative | positive) batching, for one tensor and for a tuple."""
    from refiners_b200.foundationals.latent_diffusion import StableDiffusion_1

    class Fake(fl.Module):
        def forward(self, text):
            base = torch.tensor([[float(len(t))] for t in text])
            return base, base + 0.5

    sd = StableDiffusion_1(unet=fl.Chain(fl.Identity()), clip_text_encoder=None)
    sd.clip_text_encoder = Fake()
    tokens, pooled = sd.compute_clip_text_embedding(["ab", "abcd"], ["x", ""])
    assert tokens.flatten().tolist() == [1.0, 0.0, 2.0, 4.0] and pooled.flatten().tolist() == [1.5, 0.5, 2.5, 4.5]
    sd.classifier_free_guidance = False
    assert sd.compute_clip_text_embedding("abc")[0].flatten().tolist() == [3.0]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=str)
def test_clip_text_encoder_gpu(cuda_device, dtype):
    """CLIPTextEncoderL on the kernels (causal attention on the CUDA-core flash kernel, quick GeLU, LayerNorm, GEMMs)."""
    f = load_file(str(GOLDEN / "clip_text.safetensors"))
    tower = text_tower(cuda_device, dtype)
    with no_grad():
        y = tower(f["l.tokens"])
    e_max, e_rms = rel_err(y, f["l.y"])
    if dtype == torch.float32:
        assert e_max <= 2e-4, e_max
        return
    prev, oops.FAST = oops.FAST, True
    try:
        with torch.no_grad():
            eager = oclip.text_encoder(dict(tower.state_dict()), f["l.tokens"].to(cuda_device), num_layers=12, heads=12, quick_gelu=True)
    finally:
        oops.FAST = prev
    t_max, t_rms = rel_err(eager, f["l.y"])
    print(f"\n[CLIPTextEncoderL bf16] engine max-abs {e_max:.3e} rms {e_rms:.3e} | torch-eager bf16 max-abs {t_max:.3e} rms {t_rms:.3e}")
    assert e_rms <= t_rms + 1e-3 and e_max <= 1.25 * t_max + 1e-3


def double_encode(double, f, device="cpu"):
    pooling = double.layer(("Parallel", "TextEncoderWithPooling"), fl.Chain)
    assert pooling.tokenizer.pad_token_id == 0  # the bigG tower pads with 0: its end-of-text position is unique
    l_branch = double.layer(("Parallel", "CLIPTextEncoderL"), fl.Chain)
    with no_grad():
        hidden_l = l_branch(f["l.tokens"])
        hidden_g, pooled = pooling(f["xl.tokens_g"])
    return torch.cat((hidden_l, hidden_g), dim=-1), pooled


def test_sdxl_double_text_encoder_host():
    f = load_file(str(GOLDEN / "clip_text.safetensors"))
    embedding, pooled = double_encode(double_tower("cpu", torch.float32), f)
    assert rel_err(embedding, f["xl.embedding"])[0] <= 1e-5 and rel_err(pooled, f["xl.pooled"])[0] <= 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=str)
def test_sdxl_double_text_encoder_gpu(cuda_device, dtype):
    """SDXL's DoubleTextEncoder (L + bigG towers at their penultimate layer, pooled + projected bigG embedding) on recorded
    token ids: the L tower's ids go in, the bigG tokenizer differs only in its padding id, so its ids are substituted."""
    f = load_file(str(GOLDEN / "clip_text.safetensors"))
    embedding, pooled = double_encode(double_tower(cuda_device, dtype), f)
    e1, _ = rel_err(embedding, f["xl.embedding"])
    e2, _ = rel_err(pooled, f["xl.pooled"])
    tol = 2e-4 if dtype == torch.float32 else 4e-2
    print(f"\n[DoubleTextEncoder {dtype}] embedding max-abs {e1:.3e}, pooled {e2:.3e} of max|ref|")
    assert e1 <= tol and e2 <= tol


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=str)
def test_perceiver_resampler_gpu(cuda_device, dtype):
    """IP-Adapter "plus": the PerceiverResampler (CLIP patch features -> 16 prompt tokens) on the kernels against its own host
    evaluation in fp32 (which tests/test_reference_structure.py holds bit-identical to the reference's)."""
    from refiners_b200.foundationals.latent_diffusion.perceiver import PerceiverResampler

    torch.manual_seed(4)
    model = PerceiverResampler(latents_dim=128, num_attention_layers=2, num_attention_heads=2, head_dim=64, num_tokens=16,
                               input_dim=96, output_dim=80)
    x = torch.randn(2, 257, 96)
    with no_grad():
        want = model(x)
        got = model.to(cuda_device, dtype)(x.to(cuda_device, dtype))
    e_max, _ = rel_err(got, want)
    assert e_max <= (2e-4 if dtype == torch.float32 else 3e-2), e_max

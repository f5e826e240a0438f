#!/usr/bin/env python
"""bench.py - SDXL 1024^2 bf16 denoising steps/s on N x B200 (BASELINE.json metric), all BASELINE configs.

    python bench.py --gpus 1 --steps 30 --warmup 3                 # config 2 (the headline)
    python bench.py --config 3|4|5 ...                             # LoRA + IP-Adapter | ControlLora | SAM ViT-H
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...
    python bench.py --impl reference ...      # the reference algorithm's CPU path (oracle port), host cores
    python bench.py ... --dump-outputs DIR    # also write the last timed step's outputs as DIR/<name>.npy

A "step" is one ``StableDiffusion_XL(x, step=..)`` call at latent batch 8 with classifier-free
guidance (UNet batch 16): set contexts, sigma-scale, SDXLUNet forward, CFG combine, Euler update
(BASELINE configs[1]; random-init weights, synthetic embeddings).  Config 4 uses latent batch 4 per GPU
(BASELINE configs[3]: 32 latents over 8 GPUs); config 5 is one SAM ViT-H encoder forward over a batch of
1024^2 images.  Each rank runs its own batch (weak scaling, no per-step collective; NCCL only broadcasts the
weights at init).

One JSON line is printed by rank 0: value (device-resident inputs), e2e (host buffers through the public
API, H2D/D2H inside the timed region), roofline of the dominant kernel measured live, gpu_eager_baseline
(the reference's own ATen calls - F.linear / F.conv2d / F.group_norm / SDPA - in bf16 on the same GPU, same
weights and inputs: what stock PyTorch eager delivers), cpu_baseline (oracle port on the host cores, bounded
sample), clocks, gpu_launches.  Before anything is timed, the graphed step is checked against the eager step
(bit-exact) and for finiteness.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

# SURVEY.md section 8(d): algorithmic FLOPs (2 x MAC; attention 4 B H Sq Sk d) per UNet-batch row / per image
TFLOP_PER_UNIT = {2: 6.761, 3: 6.942, 4: 9.782, 5: 5.9}
LATENT_BATCH = {2: 8, 3: 8, 4: 4, 5: 4}
METRICS = {
    2: "SDXL 1024^2 bf16 denoising steps/s (latent batch 8, CFG, Euler)",
    3: "SDXL + 2x rank-16 LoRA on every CrossAttentionBlock Linear + IP-Adapter, 1024^2 bf16 denoising steps/s (latent batch 8, CFG, Euler)",
    4: "SDXL + ControlLora 1024^2 bf16 denoising steps/s (latent batch 4 per GPU, CFG, Euler)",
    5: "SAM ViT-H image encoder 1024^2 bf16 images/s",
}
UNITS = {2: "steps/s", 3: "steps/s", 4: "steps/s", 5: "images/s"}
CL_RANK = 64  # config 4: LoRA rank inside the control copy

T0 = time.time()


def log(msg: str) -> None:
    print(f"[bench {time.time() - T0:7.1f}s] {msg}", file=sys.stderr, flush=True)


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir: str, outputs: dict[str, torch.Tensor]) -> None:
    """Write each output as ``out_dir/<name>.npy`` in float32, so that two builds can be compared output for output.
    Past DUMP_BYTES in all, each output is cut to the same fixed, seeded sample of its flattened elements."""
    import numpy as np

    path = Path(out_dir)
    path.mkdir(parents=True, exist_ok=True)
    total = 4 * sum(t.numel() for t in outputs.values())
    for name, t in outputs.items():
        values = t.detach().float().cpu()
        if total > DUMP_BYTES:
            keep = t.numel() * (DUMP_BYTES - 4096 * len(outputs)) // total
            values = values.flatten()[torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:keep].sort().values]
        np.save(path / f"{name}.npy", values.numpy())
    log(f"outputs of the last timed step written to {path}: {', '.join(outputs)}")


def measured_peaks() -> tuple[dict, str]:
    path = ROOT / "MEASURED_PEAKS.json"
    if path.exists():
        try:
            return json.loads(path.read_text()), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def usable_cores() -> int:
    """Host threads this process can really use: affinity mask and cgroup CPU quota, capped at 32
    (ATen's CPU kernels stop scaling - and oversubscribed boxes collapse - well before 128 threads)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except AttributeError:
        pass
    try:
        quota, period = Path("/sys/fs/cgroup/cpu.max").read_text().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, min(n, 32))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    FIELDS = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int) -> None:
        self.index = index
        self.rows: list[list[str]] = []
        self._stop = threading.Event()
        self._thread: threading.Thread | None = None

    def _run(self) -> None:
        while not self._stop.is_set():
            try:
                out = subprocess.run(
                    ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits"],
                    capture_output=True, text=True, timeout=5,
                ).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.splitlines()[0].split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self) -> "ClockSampler":
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()
        return self

    def __exit__(self, *exc) -> None:
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=6)

    def summary(self) -> dict:
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for name, val in zip(names, r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {
            "sm_mhz": sm[len(sm) // 2] if sm else None,
            "sm_max_mhz": max(mx) if mx else None,
            "samples": len(sm),
            "reasons": sorted(reasons),
        }


# ------------------------------------------------------------------------------ synthetic inputs
def sdxl_host_inputs(lb: int, rank: int, sigma: float, dtype: torch.dtype) -> dict[str, torch.Tensor]:
    g = torch.Generator().manual_seed(1000 + rank)
    return {
        "x": (torch.randn(lb, 4, 128, 128, generator=g) * sigma).to(dtype),
        "clip": torch.randn(2 * lb, 77, 2048, generator=g).to(dtype),
        "pooled": torch.randn(2 * lb, 1280, generator=g).to(dtype),
        "ids": torch.tensor([[1024, 1024, 0, 0, 1024, 1024]]).repeat(2 * lb, 1),
    }


def module_paths(root) -> dict[int, str]:
    return {id(m): name for name, m in root.named_modules()}


# ------------------------------------------------------------------- the reference's algorithm (baselines)
class ReferenceWorkload:
    """The oracle restatement of the same workload (oracle/: test infrastructure, used here ONLY for the
    reported baselines).  In FAST mode it makes exactly the ATen calls the reference makes
    (fluxion/layers/linear.py:9, conv.py:6, norm.py:14,52, attentions.py:29-34 of the reference), so on the
    CPU it is the reference's CPU path and on the GPU it is "PyTorch eager on a B200" - without the Chain
    walker's interpreter time, i.e. slightly favourable to the reference."""

    def __init__(self, config: int, sd: dict, extras: dict, inputs: dict[str, torch.Tensor]) -> None:
        from oracle import euler as oeuler
        from oracle import ops as oops
        from oracle import sam as osam
        from oracle import unet as ounet

        oops.FAST = True
        self.config, self.sd, self.extras, self.inp = config, sd, extras, inputs
        self.ounet, self.osam, self.oeuler = ounet, osam, oeuler
        if config != 5:
            x = inputs["x"]
            self.schedule = oeuler.EulerSchedule(30, dtype=x.dtype)
            self.schedule.timesteps = self.schedule.timesteps.to(x.device)
            self.schedule.sigmas = self.schedule.sigmas.to(x.device)

    def _unet(self, lat: torch.Tensor, ts: torch.Tensor) -> torch.Tensor:
        i, e, o = self.inp, self.extras, self.ounet
        if self.config == 4:
            deltas = o.sdxl_control_lora(e["control"], e["own"], lat, ts, i["clip"], i["pooled"], i["ids"], e["condition"], scale=e["scale"])
            return o.sdxl_unet(self.sd, lat, ts, i["clip"], i["pooled"], i["ids"], residuals=deltas)
        return o.sdxl_unet(self.sd, lat, ts, i["clip"], i["pooled"], i["ids"])

    def sliced(self, rows: int) -> "ReferenceWorkload":
        """The same workload on the first ``rows`` rows / images (shared weights): the warm-up of the CPU legs."""
        if self.config == 5:
            return ReferenceWorkload(5, self.sd, {}, {"x": self.inp["x"][:rows]})
        inp = {"x": self.inp["x"][: rows // 2], **{k: self.inp[k][:rows] for k in ("clip", "pooled", "ids")}}
        sd, extras = self.sd, dict(self.extras)
        if getattr(sd, "ip_embedding", None) is not None:
            sd = self.ounet.Weights(sd, loras=sd.loras, ip=sd.ip, ip_scale=sd.ip_scale, ip_embedding=sd.ip_embedding[:rows])
        if "condition" in extras:
            extras["condition"] = extras["condition"][:rows]
        return ReferenceWorkload(self.config, sd, extras, inp)

    def step(self, s: int) -> torch.Tensor:
        if self.config == 5:
            return self.osam.sam_vit(self.sd, self.inp["x"], num_layers=32, heads=16, global_indices=(7, 15, 23, 31))
        return self.oeuler.denoise_step(self._unet, self.schedule, self.inp["x"], s % 30, 5.0)


def reference_workload_from_model(config: int, model, extras: dict, inputs: dict[str, torch.Tensor]) -> ReferenceWorkload:
    """Same weights (shared storage), same inputs as the engine arm."""
    from oracle import unet as ounet

    if config == 3:
        sd = ounet.Weights(extras["base_sd"], loras=extras["loras"], ip=extras["ip"], ip_scale=extras["ip_scale"],
                           ip_embedding=extras["ip_embedding"])
        return ReferenceWorkload(config, sd, {}, inputs)
    if config == 4:
        ex = dict(extras, control=ounet.Weights(extras["base_sd"], loras=extras["loras"]))
        return ReferenceWorkload(config, extras["base_sd"], ex, inputs)
    return ReferenceWorkload(config, extras["base_sd"], {}, inputs)


# ------------------------------------------------------------------------------------ CPU legs
def cpu_reference(config: int, rows: int, threads: int) -> tuple[ReferenceWorkload, str]:
    """The reference's CPU path (fp32, oracle port in FAST mode) on ``rows`` UNet-batch rows / images of the
    benchmark's workload with keyed weights (oracle/cases.py)."""
    from oracle import cases
    from oracle import unet as ounet

    torch.set_num_threads(threads)
    api = cases.engine_api()  # only used to enumerate state-dict shapes / adapter layouts on the meta device
    if config == 5:
        sam = api.SAMViTH(device="meta")
        from oracle.weights import keyed_state_dict

        sd = keyed_state_dict({k: tuple(v.shape) for k, v in sam.state_dict().items()}, seed=8)
        x = cases.keyed_input("bench.cpu.images", (rows, 3, 1024, 1024))
        return ReferenceWorkload(5, sd, {}, {"x": x}), f"{rows} image(s) of 1024^2, fp32"
    assert rows % 2 == 0, "CFG rows come in (unconditional, conditional) pairs"
    lb = rows // 2
    base = cases.sdxl_base_weights(api)
    inp = {
        "x": cases.keyed_input("bench.cpu.x", (lb, 4, 128, 128)) * 14.6,
        "clip": cases.keyed_input("bench.cpu.clip", (rows, 77, 2048)),
        "pooled": cases.keyed_input("bench.cpu.pooled", (rows, 1280)),
        "ids": torch.tensor([[1024, 1024, 0, 0, 1024, 1024]]).repeat(rows, 1),
    }
    extras: dict = {}
    sd: dict = base
    if config == 3:
        unet = cases.build_sdxl(api, {k: v.to("meta") for k, v in base.items()}, "meta")
        _, ex = cases.attach_config3(api, unet, rows, "meta")
        sd = ounet.Weights(base, loras=ex["loras"], ip=ex["ip"], ip_scale=ex["ip_scale"], ip_embedding=ex["ip_embedding"])
    elif config == 4:
        unet = cases.build_sdxl(api, {k: v.to("meta") for k, v in base.items()}, "meta")
        _, ex = cases.attach_config4(api, unet, rows, "meta")
        extras = {"control": ounet.Weights(base, loras=ex["loras"]), "own": ex["own"], "condition": ex["condition"], "scale": ex["scale"]}
    what = f"latent batch {lb} + CFG (UNet batch {rows}) at 128x128 latents, fp32"
    return ReferenceWorkload(config, sd, extras, inp), what


def time_cpu(work: ReferenceWorkload, steps: int) -> float:
    with torch.no_grad():
        t0 = time.perf_counter()
        for s in range(steps):
            work.step(s)
        return (time.perf_counter() - t0) / max(steps, 1)


def run_reference_arm(args) -> None:
    """The reference's own CPU implementation of the path, on the box's host cores, through the oracle port
    (the reference package itself is pure Python over PyTorch and is not installed on the GPU box: see
    DESIGN.md).  One FULL step of the benchmark's workload (UNet batch 16 for config 2) is timed - no
    extrapolation from a smaller sample; because such a step takes about a minute on the host, the run is
    1 warm-up on a two-row batch + ``min(steps, 1)`` timed full steps and says so in the line."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = args.config
    threads = usable_cores()
    rows = args.latent_batch * 2 if cfg != 5 else args.latent_batch
    log(f"reference arm: config {cfg}, {rows} rows on {threads} host threads")
    work, _ = cpu_reference(cfg, rows, threads)
    log("reference arm: weights ready; warm-up on a two-row slice")
    time_cpu(work.sliced(2 if cfg != 5 else 1), 1)
    timed = 1
    dt = time_cpu(work, timed)
    log(f"reference arm: full step measured, {dt:.1f} s")
    units = 1 if cfg != 5 else rows
    value = units / dt
    sample = (f"{timed} full step of the workload (" + ("SAM batch %d" % rows if cfg == 5 else "UNet batch %d" % rows)
              + f"), fp32, oracle port calling the reference's ATen CPU ops, {threads} threads; measured, not extrapolated")
    line = {
        "impl": "reference",
        "metric": METRICS[cfg], "value": value, "unit": UNITS[cfg], "n_gpus": args.gpus, "steps": timed, "warmup": 1,
        "steps_requested": args.steps, "warmup_requested": args.warmup,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(cfg, args.latent_batch), "timed": sample},
        "cpu_baseline": {"value": value, "unit": UNITS[cfg], "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNITS[cfg], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def run_config1(args) -> None:
    """BASELINE config 1: SD1UNet single forward, 64x64 latent, batch 1, fp32 on the CPU - plumbing and correctness, no GPU.
    The host path of this package (leaves fall through to their torch.nn parents) is timed against the oracle port calling
    the reference's own ATen ops, on the same inputs and weights, and the two outputs are compared."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle import ops as oops
    from oracle import unet as ounet
    from oracle.weights import keyed_state_dict
    from refiners_b200.fluxion.utils import manual_seed, no_grad
    from refiners_b200.foundationals.latent_diffusion import SD1UNet

    threads = usable_cores()
    torch.set_num_threads(threads)
    manual_seed(0)
    unet = SD1UNet(in_channels=4, device="meta")
    sd = keyed_state_dict({k: tuple(v.shape) for k, v in unet.state_dict().items()}, seed=1)
    unet.load_state_dict(sd, assign=True)
    x, ctx, ts = torch.randn(1, 4, 64, 64), torch.randn(1, 77, 768), torch.tensor([[500.0]])

    def engine() -> torch.Tensor:
        unet.set_timestep(ts)
        unet.set_clip_text_embedding(ctx)
        return unet(x)

    def reference() -> torch.Tensor:
        return ounet.sd1_unet(sd, x, ts, ctx)

    prev, oops.FAST = oops.FAST, True
    try:
        with no_grad():
            repeats = args.steps
            times = {}
            for name, fn in (("engine", engine), ("reference", reference)):
                for _ in range(max(args.warmup, 1)):
                    out = fn()
                t0 = time.perf_counter()
                for _ in range(repeats):
                    out = fn()
                times[name] = ((time.perf_counter() - t0) / repeats, out)
    finally:
        oops.FAST = prev
    (t_engine, y), (t_ref, y_ref) = times["engine"], times["reference"]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"unet_output": y})
    err = float((y - y_ref).abs().max() / y_ref.abs().max())
    if not err <= 1e-5:
        raise SystemExit(f"bench.py --config 1: host path differs from the reference's ATen evaluation by {err:.3e}")
    line = {
        "metric": "SD1UNet 64x64 fp32 forwards/s on the CPU (BASELINE config 1: plumbing, no GPU)", "value": 1.0 / t_engine,
        "unit": "forwards/s", "n_gpus": 0, "steps": repeats, "warmup": max(args.warmup, 1), "ms_per_step": t_engine * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "SD1UNet(in_channels=4) fp32, x 1x4x64x64, text 1x77x768, timestep 500, one forward on the host",
                   "baseline_config": 1, "max_rel_diff_vs_reference_ops": err, "threads": threads},
        "gpu_launches": 0,
        "cpu_baseline": {"value": 1.0 / t_ref, "unit": "forwards/s", "cores": threads, "kind": "port",
                         "sample": f"{repeats} full forwards of the same workload through the oracle port (the reference's ATen CPU ops)"},
        "e2e": {"value": 1.0 / t_engine, "unit": "forwards/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_name(cfg: int, lb: int) -> str:
    if cfg == 5:
        return f"SAMViTH image encoder, {lb} x 3 x 1024 x 1024 per GPU, bf16"
    extra = {2: "", 3: " + 700 LoRA adapters (2 x rank 16) + SDXL IP-Adapter (4 image tokens)",
             4: f" + ControlLora('canny', rank-{CL_RANK} LoRAs in the control copy)"}[cfg]
    return f"SDXLUNet 1024^2 bf16{extra}, 30-step Euler, latent batch {lb} + CFG (UNet batch {2 * lb}) per GPU"


# ------------------------------------------------------------------------------------ GPU arm
def dominant_kernel_roofline(device: torch.device, peaks: dict, peaks_kind: str, cfg: int, lb: int) -> dict:
    """tc_gemm on the most frequent GEMM of the workload, timed alone with CUDA events, L2 flushed between
    launches.  SDXL: [B*1024, 1280] x [1280, 1280]^T (240 of 743 Linear calls per forward, SURVEY 8a A2);
    SAM: the MLP up-projection [B*4096, 1280] x [5120, 1280]^T with its bias + GeLU epilogue."""
    from refiners_b200 import backend as B

    if cfg == 5:
        M, K, N = lb * 4096, 1280, 5120
    else:
        M, K, N = 2 * lb * 1024, 1280, 1280
    x = torch.randn(M, K, device=device, dtype=torch.bfloat16)
    w = torch.randn(N, K, device=device, dtype=torch.bfloat16) * 0.03
    flush = torch.empty(256 * 1024 * 1024, device=device, dtype=torch.uint8)
    if cfg == 5:  # as the encoder launches it: bias + GeLU in the epilogue
        bias = torch.randn(N, device=device, dtype=torch.bfloat16)
        launch = lambda: B.linear(x, w, bias, epilogue=B.EPI_GELU)  # noqa: E731
    else:
        launch = lambda: B.linear(x, w)  # noqa: E731
    with torch.no_grad():
        for _ in range(5):
            launch()
        torch.cuda.synchronize()
        times = []
        for _ in range(20):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            launch()
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
    ms = sum(times) / len(times)
    ms_median = sorted(times)[len(times) // 2]
    flops = 2.0 * M * N * K
    achieved = flops / (ms * 1e-3) / 1e12
    peak = float(peaks["bf16_tflops"])
    # dram__bytes_read.sum + dram__bytes_write.sum of this kernel on this shape from this round's `ncu --set full`
    # capture (tools/ncu_summary.py writes the json next to the text summary); null when no capture is committed
    traffic, traffic_source = None, None
    cap = ROOT / "profiles" / "r02_ncu_gemm_dominant.json"
    if cfg != 5 and cap.exists():
        try:
            rec = json.loads(cap.read_text())
            if rec.get("shape") == [M, N, K]:
                traffic, traffic_source = float(rec["dram_bytes"]), f"profiles/{cap.name}"
        except Exception:
            pass
    return {
        "bound": "tensor", "kernel": f"tc_gemm_kernel<bf16, cta_group::2 pair> [{M}x{K}]x[{K}x{N}]^T" + (" + bias + GeLU" if cfg == 5 else ""),
        "achieved": achieved,
        "peak": peak, "peak_source": f"{peaks_kind} bf16_tflops (burst: kernel timed alone)", "unit": "TFLOP/s",
        "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_source, "ms_per_launch": ms, "ms_per_launch_median": ms_median,
        "algorithmic_flops_per_launch": flops, "algorithmic_bytes_per_launch": 2.0 * (M * K + N * K + M * N),
    }


def build_sdxl_workload(cfg: int, device: torch.device, dtype: torch.dtype, lb: int, world: int):
    """The engine arm's model for configs 2-4, plus the description the baselines need (paths of the adapted
    leaves recorded before injection; tensors are the model's own)."""
    import refiners_b200.fluxion.layers as fl
    from refiners_b200.fluxion.adapters import LinearLora, LoraAdapter
    from refiners_b200.foundationals.latent_diffusion import Euler, SDXLUNet, StableDiffusion_XL

    unet = SDXLUNet(in_channels=4, device=device, dtype=dtype)
    extras: dict = {"base_sd": dict(unet.state_dict())}
    if cfg == 3:
        from refiners_b200.foundationals.clip.image_encoder import CLIPImageEncoderH
        from refiners_b200.foundationals.latent_diffusion.cross_attention import CrossAttentionBlock
        from refiners_b200.foundationals.latent_diffusion.image_prompt import SDXLIPAdapter

        paths = module_paths(unet)
        targets = [
            (lin, parent) for lin, parent in unet.walk(fl.Linear, recurse=True)
            if any(isinstance(a, CrossAttentionBlock) for a in [*parent.get_parents(), parent])
        ]
        cross = {id(a): paths[id(a)] for a in unet.layers(fl.Attention) if type(a) is not fl.SelfAttention}
        loras: dict = {}
        for lin, parent in targets:
            mods = []
            for j, scale in enumerate((1.0, 1.4)):
                lora = LinearLora(f"lora{j}", in_features=lin.in_features, out_features=lin.out_features, rank=16, scale=scale,
                                  device=device, dtype=dtype)
                lora.up.weight.data.normal_(0, 0.02)  # re-drawn: the default zero init would make the LoRA work a multiply by zero
                mods.append(lora)
                loras.setdefault(paths[id(lin)], []).append((lora.down.weight, lora.up.weight, scale))
            LoraAdapter(lin, *mods).inject(parent)
        ip = SDXLIPAdapter(unet, clip_image_encoder=CLIPImageEncoderH(device="meta"), scale=0.6)
        ip.inject()
        emb = torch.randn(2 * lb, 4, 2048, device=device, dtype=dtype)
        ip.set_clip_image_embedding(emb)
        extras.update(loras=loras, ip={cross[id(s.target)]: (s.image_key_projection.weight, s.image_value_projection.weight) for s in ip.sub_adapters},
                      ip_scale=0.6, ip_embedding=emb, adapters=len(targets), keep=ip)
    elif cfg == 4:
        from refiners_b200.foundationals.latent_diffusion.stable_diffusion_xl.control_lora import ControlLoraAdapter, ZeroConvolution

        adapter = ControlLoraAdapter("canny", unet, scale=1.0)
        cl = adapter.control_lora
        for zc in cl.layers(ZeroConvolution):
            for prm in zc.parameters():
                prm.data.normal_(0, 0.02)  # zero-initialised by design: re-drawn so the control path does real work
        own = dict(cl.state_dict())
        paths = module_paths(cl)
        g = torch.Generator().manual_seed(7)
        sd, loras = {}, {}
        for lin, _ in cl.walk(fl.Linear, recurse=True):
            down = (torch.randn(CL_RANK, lin.in_features, generator=g) / CL_RANK).to(device, dtype)
            up = (torch.randn(lin.out_features, CL_RANK, generator=g) * 0.02).to(device, dtype)
            sd[f"ControlLora.{paths[id(lin)]}.down"], sd[f"ControlLora.{paths[id(lin)]}.up"] = down, up
            loras[paths[id(lin)]] = [(down, up, 1.0)]
        ControlLoraAdapter.load_lora_layers("canny", sd, cl)
        adapter.inject()
        cond = torch.rand(2 * lb, 3, 1024, 1024, device=device, dtype=dtype)
        adapter.set_condition(cond)
        extras.update(own=own, loras=loras, condition=cond, scale=1.0, adapters=len(loras), keep=adapter)
    if world > 1:  # identical replicas: weights come from rank 0 over NCCL/NVLink, once
        from refiners_b200.engine.sharding import broadcast_parameters

        broadcast_parameters(unet, src=0)
    sdxl = StableDiffusion_XL(unet=unet, solver=Euler(num_inference_steps=30), device=device, dtype=dtype)
    return sdxl, extras


def run_gpu_arm(args) -> None:
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the GPU arm has no CPU fallback; use --impl reference for the CPU path)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)

    from refiners_b200 import backend as B
    from refiners_b200.fluxion.utils import manual_seed, no_grad

    B.load_library()
    cfg, lb, dtype = args.config, args.latent_batch, torch.bfloat16
    manual_seed(0)
    log(f"building config {cfg} (random init on device)")
    runner = None
    if cfg == 5:
        from refiners_b200.foundationals.segment_anything import SAMViTH

        model = SAMViTH(device=device, dtype=dtype)
        for m in model.modules():  # rel-pos tables are zero-initialised; make them non-trivial
            if hasattr(m, "horizontal_embedding"):
                m.horizontal_embedding.data.normal_(0, 0.02)
                m.vertical_embedding.data.normal_(0, 0.02)
        if world > 1:
            from refiners_b200.engine.sharding import broadcast_parameters

            broadcast_parameters(model, src=0)
        extras = {"base_sd": dict(model.state_dict())}
        g = torch.Generator().manual_seed(1000 + rank)
        host = {"x": torch.randn(lb, 3, 1024, 1024, generator=g).to(dtype).pin_memory()}
        dev = {k: v.to(device) for k, v in host.items()}
        out_host = torch.empty(lb, 256, 64, 64, dtype=dtype).pin_memory()
        graphed = None
        if not args.no_graph and not args.profile_step:
            from refiners_b200.engine.graph import GraphedChain

            graphed = runner = GraphedChain(model)

        def forward(x: torch.Tensor) -> torch.Tensor:
            return graphed(x) if graphed is not None else model(x)

        def step_resident(s: int) -> torch.Tensor:
            return forward(dev["x"])

        def step_e2e(s: int) -> None:
            out_host.copy_(forward(host["x"].to(device, non_blocking=True)), non_blocking=True)

        def step_eager(s: int) -> torch.Tensor:
            return model(dev["x"])
    else:
        sdxl, extras = build_sdxl_workload(cfg, device, dtype, lb, world)
        host = {k: v.pin_memory() for k, v in sdxl_host_inputs(lb, rank, float(sdxl.solver.init_noise_sigma), dtype).items()}
        dev = {k: v.to(device) for k, v in host.items()}
        out_host = torch.empty_like(host["x"]).pin_memory()

        def call(x, clip, pooled, ids, s):
            return sdxl(x, step=s % 30, clip_text_embedding=clip, pooled_text_embedding=pooled, time_ids=ids)

        def step_resident(s: int) -> torch.Tensor:
            return call(dev["x"], dev["clip"], dev["pooled"], dev["ids"], s)

        def step_e2e(s: int) -> None:
            moved = {k: v.to(device, non_blocking=True) for k, v in host.items()}
            out_host.copy_(call(moved["x"], moved["clip"], moved["pooled"], moved["ids"], s), non_blocking=True)

        step_eager = step_resident
    log("model ready")
    # the dominant kernel, timed alone BEFORE the step loops heat the board into its power cap: this is the number
    # that belongs next to the burst peak (the same measurement repeated after the loops is reported beside it)
    peaks, peaks_kind = measured_peaks()
    roofline = dominant_kernel_roofline(device, peaks, peaks_kind, cfg, lb) if rank == 0 and not args.profile_step else None
    log("kernel roofline done")

    def barrier() -> None:
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    if args.profile_step:
        with no_grad():
            for s in range(2):
                step_resident(s)
            torch.cuda.synchronize()
            torch.cuda.cudart().cudaProfilerStart()
            step_resident(2)
            torch.cuda.synchronize()
            torch.cuda.cudart().cudaProfilerStop()
        print(json.dumps({"profiled_step": True, "config": cfg, "launches_in_step": B.launch_count()}), flush=True)
        return

    with no_grad():
        # ---- self-check: the timed path (graph replay) against the eager path, before anything is timed
        eager_ref = [step_eager(s).clone() for s in (0, 7)]
        if cfg != 5 and not args.no_graph:
            sdxl.enable_cuda_graph()
            runner = sdxl._graphed_unet[0]
        check = {"finite": True, "graph_equals_eager": None}
        for want, s in zip(eager_ref, (0, 7)):
            got = step_resident(s)
            check["finite"] = check["finite"] and bool(torch.isfinite(got.float()).all())
            if not args.no_graph:
                same = bool(torch.equal(got, want))
                check["graph_equals_eager"] = same if check["graph_equals_eager"] is None else (check["graph_equals_eager"] and same)
        if not check["finite"] or check["graph_equals_eager"] is False:
            raise SystemExit(f"bench.py: self-check failed before timing: {check}")
        del eager_ref
        log(f"self-check ok: {check}")

        for s in range(max(args.warmup, 3)):
            step_resident(s)
        log("warm-up done")
        launches0 = B.launch_count()
        replays0 = runner.replays if runner else 0
        barrier()
        sampler = ClockSampler(local_rank)
        with sampler:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for s in range(args.steps):
                last = step_resident(s)
            e1.record()
            barrier()
        ms_total = max_over_ranks(e0.elapsed_time(e1))
        if args.dump_outputs and rank == 0:  # before the e2e loop reuses the graph's output buffers
            dump_outputs(args.dump_outputs, {"image_embeddings" if cfg == 5 else "latents": last})
        eager_launches = B.launch_count() - launches0
        graph_launches = (runner.replays - replays0) * runner.launches_per_replay if runner else 0
        gpu_launches = eager_launches + graph_launches

        log(f"resident loop done: {ms_total / args.steps:.2f} ms/step")
        if args.resident_only:
            return
        # end to end: host buffers in, host result out, every step
        for s in range(3):
            step_e2e(s)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for s in range(args.steps):
            step_e2e(s)
        e1.record()
        barrier()
        ms_e2e = max_over_ranks(e0.elapsed_time(e1))

    units = 1 if cfg != 5 else lb
    rows = 2 * lb if cfg != 5 else lb
    ms_per_step = ms_total / args.steps
    value = world * units * 1000.0 / ms_per_step
    e2e_value = world * units * 1000.0 / (ms_e2e / args.steps)
    h2d = sum(v.numel() * v.element_size() for v in host.values())
    d2h = out_host.numel() * out_host.element_size()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    log(f"e2e loop done: {ms_e2e / args.steps:.2f} ms/step")
    after = dominant_kernel_roofline(device, peaks, peaks_kind, cfg, lb)
    sustained_peak = float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]))
    roofline["after_step_loops"] = {
        "ms_per_launch": after["ms_per_launch"], "achieved": after["achieved"], "peak": sustained_peak,
        "peak_source": f"{peaks_kind} bf16_tflops_sustained (board at its power cap)", "frac": after["achieved"] / sustained_peak,
    }
    step_tflop = TFLOP_PER_UNIT[cfg] * rows
    step_tflops = step_tflop / (ms_per_step * 1e-3)
    sustained = float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]))
    roofline_step = {
        "bound": "tensor", "achieved": step_tflops, "peak": sustained,
        "peak_source": f"{peaks_kind} bf16_tflops_sustained (kernel timed inside a long step)", "unit": "TFLOP/s",
        "frac": step_tflops / sustained, "algorithmic_tflop_per_step": step_tflop,
    }

    # ---- the competitor: the reference's ATen calls, bf16, same GPU, same weights and inputs
    eager = None
    if not args.skip_eager_baseline:
        try:
            ref_inputs = dict(dev) if cfg != 5 else {"x": dev["x"]}
            work = reference_workload_from_model(cfg, None, extras, ref_inputs)
            with torch.no_grad():
                for s in range(3):
                    out = work.step(s)
                torch.cuda.synchronize()
                n = max(3, min(args.steps, 10))
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for s in range(n):
                    out = work.step(s)
                e1.record()
                torch.cuda.synchronize()
            ms_eager = e0.elapsed_time(e1) / n
            eager = {
                "value": units * 1000.0 / ms_eager, "unit": UNITS[cfg], "ms_per_step": ms_eager, "steps": n, "dtype": "bf16",
                "what": "oracle port in FAST mode = the reference's own ATen calls (F.linear, F.conv2d, F.group_norm, F.layer_norm, "
                        "F.scaled_dot_product_attention: cuBLASLt / cuDNN / flash SDPA), same device, weights and inputs, no Chain-walker overhead",
                "finite": bool(torch.isfinite(out.float()).all()),
            }
            del work
            log(f"gpu eager baseline done: {ms_eager:.2f} ms/step")
        except Exception as exc:  # a baseline must never take the measurement down with it
            eager = {"error": f"{type(exc).__name__}: {exc}"[:300]}
            log(f"gpu eager baseline failed: {eager['error']}")

    cpu = None
    if not args.skip_cpu_baseline:
        threads = usable_cores()
        sample_rows = 4 if cfg != 5 else 1
        log(f"cpu baseline on {threads} threads (os.cpu_count() = {os.cpu_count()})")
        work, what = cpu_reference(cfg, sample_rows, threads)
        dt = time_cpu(work, 1)
        del work
        log("cpu baseline done")
        per_step = dt * rows / sample_rows  # scaled to the metric's unit by linearity in the batch (stated in `sample`)
        cpu = {"value": units / per_step, "unit": UNITS[cfg], "cores": threads, "kind": "port",
               "sample": f"one forward of {what}, oracle port calling the reference's ATen CPU ops, {dt:.1f} s measured; "
                         f"scaled x{rows // sample_rows if rows >= sample_rows else rows / sample_rows} in the batch to the metric's unit",
               "seconds_measured": dt, "rows_measured": sample_rows}

    line = {
        "metric": METRICS[cfg], "value": value, "unit": UNITS[cfg], "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {
            "workload": workload_name(cfg, lb), "baseline_config": cfg,
            "weights": "random init (seed 0), broadcast from rank 0", "cuda_graph": not args.no_graph,
            "l2": "per-step working set (weights + activations, > 5 GB) exceeds the 126 MB L2; no flush needed",
            "parallelism": f"replicas x{world} (batch-sharded, no per-step collective)",
            "self_check": check, "adapters": extras.get("adapters"),
            "launches_per_replay": runner.launches_per_replay if runner else None,
            "hoisted_step_invariant_ops": getattr(runner, "hoisted_ops", None) if runner else None,
        },
        "e2e": {"value": e2e_value, "unit": UNITS[cfg], "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": int(gpu_launches),
        "roofline": roofline,
        "roofline_step": roofline_step,
        "gpu_eager_baseline": eager,
        "vs_eager": (value / world / eager["value"]) if eager and "value" in eager else None,
        "cpu_baseline": cpu,
        "clocks": sampler.summary(),
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3, 4, 5], help="BASELINE.json configs[] index + 1 (1 = the CPU plumbing case)")
    ap.add_argument("--latent-batch", type=int, default=None, help="latents (config 5: images) per GPU; default per config")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-eager-baseline", action="store_true")
    ap.add_argument("--resident-only", action="store_true", help="stress mode: skip the e2e loop and the extras")
    ap.add_argument("--profile-step", action="store_true",
                    help="run ONE eager step between cudaProfilerStart/Stop and exit (for ncu --profile-from-start off)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32; a fixed seeded "
                         "sample when the outputs exceed 64 MB); inputs and weights are seeded, so runs with the same arguments compare")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.profile_step):
        ap.error("--dump-outputs records the timed steps of the CUDA path (or of config 1)")
    if args.config == 1:
        run_config1(args)
        return
    if args.latent_batch is None:
        args.latent_batch = LATENT_BATCH[args.config]
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()

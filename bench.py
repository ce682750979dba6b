#!/usr/bin/env python
"""bench.py — images/sec of the txt2img hot path (CFG denoising loop + VAE decode), the metric BASELINE.json names.

  python bench.py --gpus N --steps K --warmup W [--config sd15|sdxl] [--dtype bf16|fp16] [--impl sdxe|reference] [--only-headline]
                   [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch: `process_images` of B images. ONE invocation measures the whole
metric and prints ONE JSON line:
  * headline (top-level keys; BASELINE configs[1]): SD1.5 512x512, 20 Euler-a steps, B=8 per GPU, bf16;
  * "fp16": the same workload in fp16 — the reference's own arithmetic (modules/sd_hijack_unet.py:40-54);
  * "sdxl" (configs[2] / [4]): SDXL-base 1024x1024, 30 DPM++ 2M Karras steps, B=4 per GPU;
  * "c4" (configs[3]): SD1.5 512x512 + latent hires fix to 1024x1024, 20 + 20 Euler-a steps, B=4 per GPU;
  * "shard_parity": rank 0 regenerates another rank's images from its seeds / conditioning and compares the uint8 pixels
    bit for bit (N = 1: a repeated run of its own batch).
Weights are random-init of the exact architecture, conditioning is synthetic. N>1: one process per GPU (torchrun),
images sharded one block per rank, ONE NCCL broadcast of each packed weight blob at load, no per-step collective (weak
scaling). The sub-blocks time min(K, 5) steps after 2 warm-ups so that the default run stays within minutes.

Every block carries `value` (inputs resident in HBM, result left on the device) and `e2e` (same call with pinned HOST
conditioning copied in and uint8 images copied out inside the timed region); the headline and "sdxl" also carry
`roofline` of the dominant kernel class (tcgen05 GEMM / implicit-GEMM conv; per-launch CUDA-event timing from one extra
instrumented pass after the timed region), `torch_sdp_gpu` (the reference's default-SDP GPU path restated in PyTorch,
same box, same run) and `cpu_baseline` (oracle = the reference's `--use-cpu all --no-half` arithmetic on the host
cores, bounded sample). `--impl reference` times only the CPU reference arm.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

# algorithmic work (BASELINE.md §2 / SURVEY §8(d)): 2*MAC over conv / linear / QK^T / PV, no padding, no recompute
PREROLL_S = float(os.environ.get("SDXE_BENCH_PREROLL_S", "6"))  # untimed load before the timed regions (see measure_workload)
TFLOP = {
    "sd15": {"unet_sample": 0.8033, "vae": 2.515, "per_image": 34.65},
    "sdxl": {"unet_sample": 6.761, "vae": 10.47, "per_image": 416.1},
}
TFLOP["c4"] = {"unet_sample": None, "vae": 10.47, "per_image": 229.6}
WORKLOADS = {
    "sd15": dict(name="SD1.5 txt2img 512x512, 20 Euler-a steps, batch 8 per GPU", width=512, height=512, steps=20,
                 sampler="Euler a", batch=8, ctx_dim=768, adm=0, arch="sd15", hires=False),
    "sdxl": dict(name="SDXL-base txt2img 1024x1024, 30 DPM++ 2M Karras steps, batch 4 per GPU", width=1024, height=1024,
                 steps=30, sampler="DPM++ 2M", batch=4, ctx_dim=2048, adm=2816, arch="sdxl", hires=False),
    "c4": dict(name="SD1.5 txt2img 512x512 + latent hires fix to 1024x1024, 20 + 20 Euler-a steps, batch 4 per GPU", width=512,
               height=512, steps=20, sampler="Euler a", batch=4, ctx_dim=768, adm=0, arch="sd15", hires=True),
}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(tflops_sustained=d.get("bf16_tflops_sustained", 1400.0), tflops_burst=d.get("bf16_tflops", 1590.0),
                    hbm_gbs=d.get("hbm_gbs", 6650.0), source="measured (MEASURED_PEAKS.json)")
    return dict(tflops_sustained=1400.0, tflops_burst=1590.0, hbm_gbs=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=3)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------------
# the reference arm / cpu_baseline: the oracle (= reference arithmetic) on the host cores, fp32, bounded sample
# ----------------------------------------------------------------------------------------------------------------------
def effective_cores() -> int:
    """Host threads this process can really use: cpu_count capped by the affinity mask and the cgroup CPU quota
    (asking torch for 128 threads inside a container that is throttled to a few cores makes the CPU arm ~10x slower
    than it should be, which would flatter the GPU / CPU ratio)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                txt = f.read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                if q > 0:
                    with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as g:
                        n = min(n, max(1, int(q / int(g.read()) + 0.5)))
            break
        except (OSError, ValueError, IndexError):
            continue
    return max(1, n)


def cpu_reference_sample(config: str, budget_note=True) -> dict:
    """One CFG UNet call (2 samples = one sampler step of ONE image) + one VAE decode of one image, each timed WARM (a
    quarter-resolution call first, so that thread pools / oneDNN primitives exist) with the oracle's seeded weights;
    images/s is extrapolated as 1 / (unet_calls * t_step + t_decode) and labelled as such."""
    from oracle.synth import init_module_  # noqa: F401
    from oracle.unet import UNetModel, sd15_config, sdxl_config
    from oracle.vae import AutoencoderKLDecode, VAEConfig

    w = WORKLOADS[config]
    cores = effective_cores()
    torch.set_num_threads(cores)
    cfg = sd15_config() if w["arch"] == "sd15" else sdxl_config()
    h, wd = w["height"] // 8, w["width"] // 8
    with torch.no_grad():
        unet = UNetModel(cfg).eval()          # default torch init is fine for timing (dense fp32 math either way)
        t = torch.tensor([500.0, 500.0])
        ctx = torch.randn(2, 77, w["ctx_dim"])
        y = torch.randn(2, w["adm"]) if w["adm"] else None
        unet(torch.randn(2, 4, h // 4, wd // 4), t, context=ctx, y=y)  # warm-up at 1/16 of the work
        x = torch.randn(2, 4, h, wd)
        t0 = time.perf_counter()
        unet(x, t, context=ctx, y=y)
        t_step = time.perf_counter() - t0
        del unet
        vae = AutoencoderKLDecode(VAEConfig()).eval()
        vae.decode(torch.randn(1, 4, h // 4, wd // 4))
        z = torch.randn(1, 4, h, wd)
        t0 = time.perf_counter()
        vae.decode(z)
        t_dec = time.perf_counter() - t0
    ips = 1.0 / (w["steps"] * t_step + t_dec)
    return {"value": ips, "unit": "images/sec", "cores": cores, "kind": "port",
            "sample": f"1 CFG UNet call (2 samples, {t_step:.2f} s, warm) + 1 VAE decode ({t_dec:.2f} s, warm), fp32 torch CPU, "
                      f"extrapolated to {w['steps']} steps/image", "t_step_s": t_step, "t_decode_s": t_dec}


def run_reference_arm(args, rank):
    if rank != 0:
        return
    w = WORKLOADS[args.config]
    vals = []
    for _ in range(max(1, min(args.steps, 2))):  # each step is a bounded sample; keep the whole run to minutes
        r = cpu_reference_sample(args.config)
        vals.append(r)
    best = max(vals, key=lambda r: r["value"])
    line = {"impl": "reference", "metric": f"images/sec {w['name']}", "value": best["value"], "unit": "images/sec",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * w["batch"] / best["value"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": w["name"], "note": "reference --use-cpu all --no-half arithmetic (oracle port), host cores"},
            "cpu_baseline": {k: best[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": best["value"], "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------------
def build_model(arch: str, dtype, device, rank: int, world: int):
    """Random-init weights of the exact architecture. Rank 0 generates + repacks; the other ranks ingest uninitialised
    tensors (same packing => same blob layout) and receive the blob through one NCCL broadcast."""
    from sdwebui_b200 import checkpoint as C
    from sdwebui_b200 import parallel as P
    from sdwebui_b200.engine import UNetSpec, VAEDecoderEngine, VAESpec
    from sdwebui_b200.processing import SdModel
    from sdwebui_b200.sd_unet import SdxeUnet

    spec = UNetSpec.sd15() if arch == "sd15" else UNetSpec.sdxl()
    ushapes, vshapes = C.unet_param_shapes(spec), C.vae_decoder_param_shapes(VAESpec())
    if rank == 0:
        usd = C.synthetic_state_dict(ushapes, seed=0, device=device, dtype=torch.float16)
        vsd = C.synthetic_state_dict(vshapes, seed=1, device=device, dtype=torch.float16)
    else:
        usd, vsd = C.empty_state_dict(ushapes, device), C.empty_state_dict(vshapes, device)
    unet = SdxeUnet(usd, spec, dtype=dtype, device=device)
    unet.activate()
    vae = VAEDecoderEngine(VAESpec(), dtype=dtype, device=device)
    vae.load_state_dict(vsd)
    vae.finalize()
    del usd, vsd
    torch.cuda.empty_cache()
    bcast_bytes = 0
    if world > 1:
        for eng in (unet.engine, vae):
            blob = eng.weight_blob()
            P.broadcast_weight_blob(blob, src=0)
            bcast_bytes += blob.numel()
        torch.cuda.synchronize()
    model = SdModel(unet, vae, is_sdxl=(arch == "sdxl"), dtype_unet=dtype, device=device)
    return model, bcast_bytes


def make_conds(w, B, device, seed):
    g = torch.Generator().manual_seed(seed)
    c = torch.randn(B, 77, w["ctx_dim"], generator=g)
    u = torch.randn(B, 77, w["ctx_dim"], generator=g)
    if w["adm"]:
        return {"crossattn": c, "vector": torch.randn(B, w["adm"], generator=g)}, {"crossattn": u, "vector": torch.randn(B, w["adm"], generator=g)}
    return c, u


def to_dev(c, device, non_blocking=True):
    if isinstance(c, dict):
        return {k: v.to(device, non_blocking=non_blocking) for k, v in c.items()}
    return c.to(device, non_blocking=non_blocking)


def pin(c):
    if isinstance(c, dict):
        return {k: v.pin_memory() for k, v in c.items()}
    return c.pin_memory()


def nbytes(c):
    if isinstance(c, dict):
        return sum(v.numel() * v.element_size() for v in c.values())
    return c.numel() * c.element_size()


def torch_sdp_gpu_baseline(config, device, B, iters=2):
    """The reference's default-SDP GPU path restated in PyTorch (oracle under fp16 autocast + SDPA, per-image VAE
    decode), same box, same workload; random torch-init weights (timing only)."""
    from oracle.pipeline import OraclePipeline, SamplingParams
    from oracle.unet import UNetModel, sd15_config, sdxl_config
    from oracle.vae import AutoencoderKLDecode, VAEConfig

    w = WORKLOADS[config]
    cfg = sd15_config() if w["arch"] == "sd15" else sdxl_config()
    with torch.device(device):
        unet = UNetModel(cfg).half().eval()
        vae = AutoencoderKLDecode(VAEConfig()).half().eval()
    pipe = OraclePipeline(unet, vae, device, dtype_unet=torch.float16, dtype_vae=torch.float16, autocast=True)
    c, u = make_conds(w, B, device, 5)
    c, u = to_dev(c, device), to_dev(u, device)
    sp = SamplingParams(sampler=w["sampler"], steps=w["steps"], width=w["width"], height=w["height"],
                        seeds=tuple(range(1000, 1000 + B)), randn_source="GPU", scale_factor=0.13025 if w["arch"] == "sdxl" else 0.18215,
                        enable_hr=w["hires"], hr_scale=2.0, hr_second_pass_steps=w["steps"] if w["hires"] else 0, denoising_strength=0.7)
    kw = dict(y_cond=c["vector"], y_uncond=u["vector"]) if isinstance(c, dict) else {}
    cc, uu = (c["crossattn"], u["crossattn"]) if isinstance(c, dict) else (c, u)
    pipe.txt2img(sp, cc, uu, **kw)  # warm-up (cuDNN autotune etc.)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        pipe.txt2img(sp, cc, uu, **kw)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    del pipe, unet, vae
    torch.cuda.empty_cache()
    return {"value": B / (ms / 1000.0), "unit": "images/sec", "ms_per_step": ms,
            "how": "oracle restatement under torch.autocast(fp16) + F.scaled_dot_product_attention, per-image VAE decode"}


def class_table(prof):
    return {k: {"ms": round(v["ms"], 4), "tflops": (v["flops"] / (v["ms"] / 1e3) / 1e12 if v["ms"] > 0 else 0),
                "gbs": (v["bytes"] / (v["ms"] / 1e3) / 1e9 if v["ms"] > 0 else 0), "launches": v["launches"]} for k, v in prof.items()}


def dump_outputs(dump_dir, outputs):
    """Writes each array as DIR/<name>.npy in float32 (uint8 pixels convert exactly). The largest workload's images
    (SDXL or hires fix, 4 x 1024 x 1024 x 3) come to 48 MiB, so every output is stored whole."""
    os.makedirs(dump_dir, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(dump_dir, f"{name}.npy"), t.float().numpy())


def measure_workload(key, dtype_name, rank, world, local, device, steps, warmup, want_roofline, want_extras, want_parity, clock_sampler=None,
                     dump_dir=None):
    """Builds the model, runs W warm-ups, times K resident steps and K end-to-end steps (max over ranks, barrier + device
    sync on both sides), optionally the roofline pass / baselines / shard-parity check. Returns the JSON block (rank 0) or None.
    With `dump_dir`, rank 0 writes what the last timed resident step returned for its own shard: `images` [B, H, W, 3]
    and `latents` [B, 4, h, w]."""
    import torch.distributed as dist

    from sdwebui_b200 import lib as L
    from sdwebui_b200 import parallel as P
    from sdwebui_b200.processing import StableDiffusionProcessingTxt2Img, process_images

    w = WORKLOADS[key]
    dtype = torch.bfloat16 if dtype_name == "bf16" else torch.float16
    B = w["batch"]
    model, bcast_bytes = build_model(w["arch"], dtype, device, rank, world)
    lib = L.load()

    def seeds_of(r):
        return [1000 + r * B + i for i in range(B)]  # global image index -> seed: sharding is invisible in the output

    c_host, u_host = make_conds(w, B, device, 7 + rank)
    c_host, u_host = pin(c_host), pin(u_host)
    c_dev, u_dev = to_dev(c_host, device, False), to_dev(u_host, device, False)
    hr = dict(enable_hr=True, hr_scale=2.0, hr_second_pass_steps=w["steps"], denoising_strength=0.7) if w["hires"] else {}

    def make_p(c, u, seeds, **kw):
        return StableDiffusionProcessingTxt2Img(sd_model=model, c=c, uc=u, seeds=seeds, sampler_name=w["sampler"], steps=w["steps"],
                                                cfg_scale=7.0, width=w["width"], height=w["height"], randn_source="GPU", **hr, **kw)

    def step_resident():
        return process_images(make_p(c_dev, u_dev, seeds_of(rank)), to_host=False)

    def step_e2e():
        return process_images(make_p(to_dev(c_host, device), to_dev(u_host, device), seeds_of(rank)), to_host=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = lib.sdxe_launch_count()
        e0.record()
        for _ in range(k):
            out = fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            tms = torch.tensor([ms], device=device)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            ms = tms.item()
        return ms, lib.sdxe_launch_count() - n0, out

    for _ in range(warmup):
        step_resident()
    step_e2e()
    # untimed pre-roll: under the 1 kW power cap the SM clock settles ~4-5 % below its cold value over the first seconds
    # of load; without it the first timed region (`value`) runs on a colder GPU than the second (`e2e`) and the two differ
    # by drift, not by the host copies (interleaved A/B: 393.1 vs 395.7 ms per batch, tools/profile_pipeline.py)
    torch.cuda.synchronize()
    t_roll, n_roll = time.perf_counter(), 0
    while time.perf_counter() - t_roll < PREROLL_S:
        step_resident()
        torch.cuda.synchronize()
        n_roll += 1
    if clock_sampler is not None:
        clock_sampler.start()
    ms_res, launches, last = timed(step_resident, steps)
    # copied to the host before the next timed region can reuse the device buffers
    outputs = {"images": last.images.cpu(), "latents": last.latents.cpu()} if dump_dir and rank == 0 else None
    ms_e2e, _, _ = timed(step_e2e, steps)
    clocks = clock_sampler.stop() if clock_sampler is not None else None
    if outputs is not None:
        dump_outputs(dump_dir, outputs)

    # ---- shard parity: rank 0 regenerates the LAST rank's images (N = 1: its own, a second time) and compares pixels
    parity = None
    if want_parity:
        mine = process_images(make_p(c_dev, u_dev, seeds_of(rank)), to_host=True).images
        gathered = P.gather_images(mine, world)
        if rank == 0:
            other = world - 1
            co, uo = make_conds(w, B, device, 7 + other)
            again = process_images(make_p(to_dev(co, device, False), to_dev(uo, device, False), seeds_of(other)), to_host=True).images
            parity = {"equal": bool(torch.equal(again, gathered[other])), "rank_checked": other,
                      "how": ("rank 0 regenerated rank %d's %d images from their seeds / conditioning; uint8 pixels compared bit for bit" % (other, B))
                      if world > 1 else "single GPU: the batch generated twice; uint8 pixels compared bit for bit"}

    n_img = B * world * steps
    block = None
    if rank == 0:
        value, e2e = n_img / (ms_res / 1000.0), n_img / (ms_e2e / 1000.0)
        peaks = load_peaks()
        block = {"metric": f"images/sec {w['name']}", "value": value, "unit": "images/sec", "n_gpus": world, "steps": steps, "warmup": warmup,
                 "ms_per_step": ms_res / steps, "dtype": dtype_name,
                 "config": {"workload": w["name"], "global_batch": B * world, "parallelism": f"dp{world} (image shards, no per-step collective)",
                            "l2": "working set (>= 1.7 GB weights + activations) >> 126 MB L2: no explicit flush",
                            "weights": "random-init, exact architecture", "weight_broadcast_bytes": bcast_bytes,
                            "preroll": f"{n_roll} untimed steps (>= {PREROLL_S:.0f} s of load) after the {warmup} warm-ups: both timed regions at settled clocks"},
                 "e2e": {"value": e2e, "unit": "images/sec", "h2d_bytes_per_step": nbytes(c_host) + nbytes(u_host),
                         "d2h_bytes_per_step": B * w["height"] * w["width"] * 3 * (4 if w["hires"] else 1), "ms_per_step": ms_e2e / steps},
                 "gpu_launches": int(launches), "clocks": clocks,
                 "whole_job_frac": value * TFLOP[key]["per_image"] / (world * peaks["tflops_sustained"]),
                 "tflop_per_image": TFLOP[key]["per_image"]}
        if parity is not None:
            block["shard_parity"] = parity["equal"]
            block["shard_parity_detail"] = parity
        if want_roofline:
            # ---- roofline of the dominant kernel class: one instrumented UNet call (2B CFG batch) + one VAE decode batch
            unet_e, vae_e = model.unet.engine, model.vae
            h, wd = w["height"] // 8, w["width"] // 8
            x = torch.randn(2 * B, 4, h, wd, device=device, dtype=dtype)
            t = torch.full((2 * B,), 500.0, device=device, dtype=dtype)
            ctx = torch.randn(2 * B, 77, w["ctx_dim"], device=device, dtype=dtype)
            y = torch.randn(2 * B, w["adm"], device=device, dtype=dtype) if w["adm"] else None
            unet_e.profile(True)
            unet_e.forward(x, t, ctx, y)
            torch.cuda.synchronize()
            prof_u = unet_e.profile_read()
            unet_e.profile(False)
            vae_e.profile(True)
            vae_e.decode(torch.randn(B, 4, h, wd, device=device, dtype=dtype))
            torch.cuda.synchronize()
            prof_v = vae_e.profile_read()
            vae_e.profile(False)
            mm_ms = prof_u["gemm"]["ms"] + prof_u["conv3x3"]["ms"]
            mm_fl = prof_u["gemm"]["flops"] + prof_u["conv3x3"]["flops"]
            mm_n = prof_u["gemm"]["launches"] + prof_u["conv3x3"]["launches"]
            achieved = mm_fl / (mm_ms / 1000.0) / 1e12 if mm_ms > 0 else 0.0
            total_u = sum(v["ms"] for v in prof_u.values())
            traffic, traffic_src = None, None
            tpath = os.path.join(ROOT, "profiles", "r2_gemm_traffic.json")   # final-tree capture; the round-1 one is the fallback
            if not os.path.exists(tpath):
                tpath = os.path.join(ROOT, "profiles", "r1c_gemm_traffic.json")
            if key == "sd15" and os.path.exists(tpath):  # ncu capture of the same kernel on the same UNet call (SD1.5, 2B = 16)
                with open(tpath) as f:
                    tj = json.load(f)
                traffic = tj["traffic_per_launch_bytes"]
                traffic_src = tj["source"] + " — a constant from that committed capture, not re-measured by this run"
            block["roofline"] = {
                "bound": "tensor", "kernel": "sdxe::gemm_kernel (tcgen05 GEMM + implicit-GEMM conv3x3)", "achieved": achieved,
                "peak": peaks["tflops_sustained"], "unit": "TFLOP/s", "frac": achieved / peaks["tflops_sustained"],
                "peak_source": peaks["source"] + ", bf16 sustained (kernel timed inside a long step)", "traffic": traffic,
                "traffic_unit": "bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum, ncu)", "traffic_source": traffic_src,
                "algorithmic_bytes_per_launch": (prof_u["gemm"]["bytes"] + prof_u["conv3x3"]["bytes"]) / max(1, mm_n),
                "launches_per_unet_call": mm_n, "avg_launch_us": 1000.0 * mm_ms / max(1, mm_n),
                "share_of_unet_call": mm_ms / total_u if total_u else None,
                "how": "CUDA events around every launch of one extra instrumented UNet call on the launching stream (sdxe_profile), "
                       "algorithmic 2*M*N*K per launch",
                "by_kernel_class_unet": class_table(prof_u), "by_kernel_class_vae": class_table(prof_v),
                "whole_job_frac": block["whole_job_frac"]}
    model.unet.deactivate()
    model.vae.close()
    del model
    torch.cuda.empty_cache()
    if rank == 0 and want_extras:
        try:
            block["torch_sdp_gpu"] = torch_sdp_gpu_baseline(key, device, B)
        except Exception as ex:  # noqa: BLE001
            block["torch_sdp_gpu"] = {"unavailable": repr(ex)[:200]}
        try:
            cb = cpu_reference_sample(key)
            block["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        except Exception as ex:  # noqa: BLE001
            block["cpu_baseline"] = {"value": None, "unit": "images/sec", "cores": effective_cores(), "kind": "port", "sample": repr(ex)[:200]}
    return block


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="sdxe", choices=["sdxe", "reference"])
    ap.add_argument("--config", default=os.environ.get("SDXE_BENCH_CONFIG", "sd15"), choices=["sd15", "sdxl", "c4"],
                    help="the workload reported at the top level of the JSON line (default: BASELINE configs[1])")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp16"])
    ap.add_argument("--no-extras", action="store_true", help="skip cpu_baseline / torch-SDP legs")
    ap.add_argument("--only-headline", action="store_true", help="skip the fp16 / sdxl / c4 blocks")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the headline's last timed step returned as DIR/<name>.npy (float32); "
                         "weights, conditioning and noise are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the sdxe path's outputs; the reference arm only times a CPU sample")

    from sdwebui_b200 import parallel as P

    world_env = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        rank = int(os.environ.get("RANK", "0"))
        run_reference_arm(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl sdxe needs a CUDA device (no CPU fallback)")
    rank, world, local = P.init_from_env("nccl" if world_env > 1 else None)
    device = torch.device(f"cuda:{local}")
    torch.cuda.set_device(device)
    import torch.distributed as dist

    extras = not args.no_extras
    warm = max(3, args.warmup)
    sampler = ClockSampler(local) if rank == 0 else None
    head = measure_workload(args.config, args.dtype, rank, world, local, device, args.steps, warm, True, extras, True, sampler,
                            args.dump_outputs)
    blocks = {}
    if not args.only_headline:
        sub_steps = max(1, min(args.steps, 5))
        other_dtype = "fp16" if args.dtype == "bf16" else "bf16"
        blocks[other_dtype] = measure_workload(args.config, other_dtype, rank, world, local, device, sub_steps, 3, False, False, False)
        for key in ("sd15", "sdxl", "c4"):
            if key == args.config:
                continue
            blocks[key] = measure_workload(key, args.dtype, rank, world, local, device, min(sub_steps, 3) if key == "c4" else sub_steps, 3,
                                           key == "sdxl", extras and key == "sdxl", key == "sdxl")
    if rank == 0:
        line = dict(head)
        line.update({"higher_is_better": True, "scaling": "weak", "vs_baseline": None, "data": "synthetic"})
        for k, blk in blocks.items():
            if blk is not None:
                line[k] = blk
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Benchmark of the AudioGPT generative hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload hifigan|ddim]
                    [--dump-outputs DIR]

--dump-outputs DIR writes what the timed GPU path returned in its last timed step, rank 0's batch, as float32 .npy
files: hifigan_wav.npy ([8, 1, 204800] waveforms) and ddim_latent.npy ([4, 4, 10, 78] DDIM end points).  Inputs and
weights are seeded, so two builds run with the same arguments can be compared output for output.

BASELINE.json's metric has two halves; one JSON line carries both:

* top level  -- mel-frames/s vocoded: HiFi-GAN V1 (22.05 kHz, hop 256) on a batch of 8 synthetic 80-bin mels of
  800 frames per GPU (BASELINE configs[1], what `FastSpeech2 TTS -> HiFi-GAN, batch 8` hands to the vocoder).
  A step is one pass of that batch through `HifiGanGenerator.forward`.
* "ddim"     -- clips/s of Make-An-Audio DDIM-100 with classifier-free guidance 1.5 on the C4 shard
  (BASELINE configs[3]: 32 ten-second clips over 8 GPUs = 4 clips, CFG batch 8, per GPU): every rank runs the
  whole 100-step chain for its 4 clips, timed on the device, max over ranks; the object has the same fields as
  the top level (value, ms_per_step, e2e, roofline, gpu_launches, config).  `--workload ddim` prints that object
  as the line itself.

  value     : device-resident inputs, CUDA-event timed, barrier + synchronize on both sides, max over ranks
  e2e       : the same metric through the public host-buffer call (pinned H2D of the inputs, D2H of the result
              inside the timed region): agpt_hifigan_vocode_host / DDIMSampler.sample on host tensors
  roofline  : the tcgen05 tap-GEMM against the measured bf16/fp16 tensor peak (MEASURED_PEAKS.json).  `frac` is
              on ALGORITHMIC FLOPs (SURVEY.md 8d: 0.614 GFLOP per mel frame, 18.66 TFLOP per clip); `frac_issued`
              counts the three fp16 products the error-compensated arithmetic issues per MAC.
  cpu_baseline / --impl reference : the CPU oracle (oracle/*.py: the reference's forward restated on torch's own
              fp32 CPU kernels -- the reference is pure Python and does not travel to the GPU box) on the host cores
  extra     : DiffSinger C3 chain (16 utt x 400 frames x 100 p_sample steps), BigVGAN base, each one full run

With N > 1 (torchrun, one rank per GPU) every rank works on its own batch (weak scaling, no data-path
collective); weights are broadcast once from rank 0; finished waveforms are all-gathered on NCCL's stream while
the next batch is computed (the gather of step i overlaps step i+1; the last one is inside the timed region).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

B_PER_GPU, T_FRAMES, HOP, SR = 8, 800, 256, 22050
METRIC, UNIT = "mel_frames_per_s_vocoded", "frames/s"
WORKLOAD = "HiFi-GAN V1 22.05kHz vocoder, batch 8 x 800 mel frames per GPU (FastSpeech2->HiFi-GAN, BASELINE configs[1])"
ARITH = "3xfp16-split: x = hi + lo fp16 parts, products hi*hi + lo*hi + hi*lo on tcgen05 kind::f16, fp32 accumulate in TMEM"

DDIM_B, DDIM_S, DDIM_SCALE, DDIM_SHAPE = 4, 100, 1.5, (4, 10, 78)
DDIM_METRIC, DDIM_UNIT = "clips_per_s_ddim100_cfg", "clips/s"
DDIM_WORKLOAD = ("Make-An-Audio txt2audio UNet (160 M params), DDIM-100, eta 0, CFG 1.5, 10 s clips (latent 4x10x78), "
                 "4 clips per GPU = the 32-clips-over-8-GPUs shard of BASELINE configs[3]")
DDIM_TFLOP_PER_CLIP = 18.66          # SURVEY.md 8d: 200 UNet forwards x 93.3 GFLOP


def base_config(n_gpus):
    return {"workload": WORKLOAD, "batch_per_gpu": B_PER_GPU, "frames_per_utt": T_FRAMES,
            "global_batch": B_PER_GPU * n_gpus, "hop": HOP, "sample_rate": SR,
            "weights": "seeded random (specs.synth_hifigan(HIFIGAN_V1, 1234))", "arith": ARITH,
            "parallelism": f"batch-sharded x{n_gpus}, no data-path collective",
            "l2_policy": "activation working set per step ~2.5 GB >> 126 MB L2 (no explicit flush needed)"}


def ddim_config(n_gpus):
    return {"workload": DDIM_WORKLOAD, "clips_per_gpu": DDIM_B, "global_batch": DDIM_B * n_gpus, "ddim_steps": DDIM_S,
            "cfg_scale": DDIM_SCALE, "latent": list(DDIM_SHAPE), "context": [77, 1024],
            "weights": "seeded random (specs.synth_unet(UNET_TXT2AUDIO, 4040))", "arith": ARITH,
            "parallelism": f"clips sharded x{n_gpus}, no data-path collective",
            "l2_policy": "weights 641 MB fp32 (1.28 GB as fp16 hi/lo images) re-read every forward >> 126 MB L2"}


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write every tensor of ``arrays`` as <out_dir>/<name>.npy in float32."""
    host = {k: v.detach().to("cpu", torch.float32).numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    assert total <= DUMP_MAX_BYTES, f"outputs to dump are {total} bytes, more than {DUMP_MAX_BYTES}"
    os.makedirs(out_dir, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


# ------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-i", str(self.gpu), "-lms", "25"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for n, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if sm:
            hi = [v for v in sm if v >= 0.5 * max(sm)]   # samples under load
            out = {"sm_mhz": statistics.median(hi), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                   "samples": len(sm)}
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


# ------------------------------------------------------------------------------------ CPU arms
_ALLOC_NOTE = ""


def _cpu_allocator_tuning():
    """The CPU forward allocates and frees 50-MB intermediates; with glibc's defaults every one of them is mmap'ed,
    page-faulted and unmapped again, which on a 128-CPU box costs the 16-thread CPU path 5x (measured: 473 -> 2 500
    frames/s, profiles/r2s_reference_arm.txt).  Keep freed memory in the heap instead (what MALLOC_MMAP_MAX_=0
    MALLOC_TRIM_THRESHOLD_=... would do from the environment): the CPU arms get their best."""
    global _ALLOC_NOTE
    if _ALLOC_NOTE:
        return
    try:
        import ctypes
        libc = ctypes.CDLL("libc.so.6")
        M_TRIM_THRESHOLD, M_TOP_PAD, M_MMAP_MAX = -1, -2, -4
        ok = libc.mallopt(M_MMAP_MAX, 0) and libc.mallopt(M_TRIM_THRESHOLD, 2**31 - 1) and libc.mallopt(M_TOP_PAD, 1 << 30)
        _ALLOC_NOTE = "glibc mallopt(M_MMAP_MAX=0, M_TRIM_THRESHOLD=2 GiB, M_TOP_PAD=1 GiB)" if ok else "glibc defaults (mallopt refused)"
    except Exception as e:                      # noqa: BLE001
        _ALLOC_NOTE = f"glibc defaults ({e!r})"


def _calibrate_threads(fn):
    """torch's intra-op pool scales badly past a few dozen threads on these convs (and torchrun pins
    OMP_NUM_THREADS=1): time a short sample at several thread counts and keep the best."""
    ncpu = os.cpu_count() or 1
    best, cores = None, ncpu
    for nt in sorted({ncpu, max(1, ncpu // 2), 64, 32, 16, 8}):
        if nt > ncpu:
            continue
        torch.set_num_threads(nt)
        fn()
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, cores = dt, nt
    torch.set_num_threads(cores)
    return cores


def cpu_vocode_rate(steps, warmup, batch, frames):
    """frames/s of the CPU oracle (the reference's forward restated on torch fp32 CPU ops)."""
    from audiogpt_b200 import specs
    from oracle import hifigan_ref as hr
    _cpu_allocator_tuning()
    h = specs.HIFIGAN_V1
    sd = specs.synth_hifigan(h, 1234)
    cal = specs.synth_tensor((1, 80, 200), seed=1, scale=2.0, shift=-4.0)
    cores = _calibrate_threads(lambda: hr.hifigan_forward(sd, h, cal))
    mel = specs.synth_tensor((batch, 80, frames), seed=0, scale=2.0, shift=-4.0)
    for _ in range(warmup):
        hr.hifigan_forward(sd, h, mel)
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        hr.hifigan_forward(sd, h, mel)
        ts.append(time.perf_counter() - t0)
    sec = sum(ts) / len(ts)
    return batch * frames / sec, sec, cores


def cpu_ddim_rate(n_steps_sample):
    """clips/s of the CPU oracle DDIM-100 + CFG chain at B = 1, from a bounded sample of its 100 steps."""
    from audiogpt_b200 import specs
    from oracle import ldm_ref as lr
    _cpu_allocator_tuning()
    cfg = specs.UNET_TXT2AUDIO
    sd = specs.synth_unet(cfg, 4040)
    tab = lr.ldm_schedule()
    x = torch.tensor(np.random.RandomState(55).randn(1, *DDIM_SHAPE), dtype=torch.float32)
    c = specs.synth_tensor((1, 77, 1024), seed=5)
    uc = specs.synth_tensor((1, 77, 1024), seed=6)
    eps = lambda a, t, ctx: lr.unet_forward(sd, cfg, a, t, ctx)
    cores = _calibrate_threads(lambda: lr.ddim_sample(eps, tab["alphas_cumprod"], DDIM_S, x, c, uc, DDIM_SCALE, steps_limit=1))
    t0 = time.perf_counter()
    lr.ddim_sample(eps, tab["alphas_cumprod"], DDIM_S, x, c, uc, DDIM_SCALE, steps_limit=n_steps_sample)
    sec_per_step = (time.perf_counter() - t0) / n_steps_sample
    return 1.0 / (sec_per_step * DDIM_S), sec_per_step, cores


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if os.environ.get("AGPT_REF_CUDA_INIT") == "1" and torch.cuda.is_available():    # diagnostic: process state of the GPU arm
        torch.zeros(1).cuda()
    if args.workload == "ddim":
        rate, sps, cores = cpu_ddim_rate(max(2, min(args.steps, 6)))
        sample = (f"B=1: {max(2, min(args.steps, 6))} of the {DDIM_S} DDIM steps (2 UNet forwards each, CFG) on {cores} threads; "
                  f"clips/s = 1 / (s_per_step x {DDIM_S})")
        line = {"impl": "reference", "metric": DDIM_METRIC, "value": rate, "unit": DDIM_UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": sps * 1e3, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": ddim_config(args.gpus),
                "cpu_baseline": {"value": rate, "unit": DDIM_UNIT, "cores": cores, "kind": "port", "sample": sample},
                "e2e": {"value": rate, "unit": DDIM_UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0, "note": "ms_per_step is one DDIM step of the sample, not one chain"}
        print(json.dumps(line))
        return
    # bounded sample of the same workload: 2 of the 8 utterances per step (same T) in one forward call, as the
    # reference would run them; the RATE is the result, ms_per_step is the sample's own (not extrapolated)
    sb = 2
    rate, sec, cores = cpu_vocode_rate(args.steps, max(1, min(args.warmup, 2)), sb, T_FRAMES)
    sample = f"{sb} of {B_PER_GPU} utterances x {T_FRAMES} frames per step ({sb * T_FRAMES} frames), {args.steps} steps, {cores} threads; {_ALLOC_NOTE}"
    ddim_rate, ddim_sps, ddim_cores = cpu_ddim_rate(3)
    line = {"impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "frames_per_step": sb * T_FRAMES,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": base_config(args.gpus),
            "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "ddim": {"impl": "reference", "metric": DDIM_METRIC, "value": ddim_rate, "unit": DDIM_UNIT,
                     "cpu_baseline": {"value": ddim_rate, "unit": DDIM_UNIT, "cores": ddim_cores, "kind": "port",
                                      "sample": f"B=1: 3 of the {DDIM_S} DDIM steps (CFG pair per step); clips/s = 1/(s_per_step x {DDIM_S})"},
                     "s_per_ddim_step": ddim_sps},
            "note": "CPU oracle port of HifiGanGenerator.forward / DDIMSampler+UNetModel (the reference is pure PyTorch and "
                    "/root/reference does not travel to the GPU box, so kind = port); ms_per_step and frames_per_step "
                    "describe the bounded sample actually run; RTF = value*hop/sample_rate"}
    line["x_realtime"] = rate * HOP / SR
    print(json.dumps(line))


# ------------------------------------------------------------------------------------ GPU arm: DDIM (C4)
def measure_ddim(dev, rank, n_gpus, chains, peaks, want_cpu, keep=None, outputs=None):
    """All ranks: DDIM-100 + CFG for DDIM_B clips per rank.  Returns the 'ddim' object (rank 0) or None.
    ``keep`` (a dict) receives the sampler so that the mixed-dispatch measurement can reuse the 160 M-param engine;
    ``outputs`` (a dict) receives the latent of the last timed chain as 'ddim_latent'."""
    import ctypes as C
    import torch.distributed as dist
    from audiogpt_b200 import _lib, parallel, specs
    from audiogpt_b200.ldm.models.diffusion.ddim import DDIMSampler, LatentDiffusionShim
    from audiogpt_b200.ldm.modules.diffusionmodules.openaimodel import UNetModel

    cfg = specs.UNET_TXT2AUDIO
    shapes = specs.unet_param_shapes(cfg)
    sd = specs.synth_unet(cfg, 4040) if rank == 0 else {k: torch.empty(s) for k, s in shapes.items()}
    sd = parallel.broadcast_state_dict(sd, src=0)
    u = UNetModel(image_size=32, use_checkpoint=True, **cfg)
    u.load_state_dict(sd, strict=True)
    del sd
    u = u.eval().to(dev)
    smp = DDIMSampler(LatentDiffusionShim(u).to(dev))
    B = DDIM_B
    xT_h = torch.tensor(np.random.RandomState(55 + rank).randn(B, *DDIM_SHAPE), dtype=torch.float32).pin_memory()
    c_h = specs.synth_tensor((B, 77, 1024), seed=5 + 10 * rank).pin_memory()
    uc_h = specs.synth_tensor((1, 77, 1024), seed=6).expand(B, -1, -1).contiguous().pin_memory()
    xT, c, uc = xT_h.to(dev), c_h.to(dev), uc_h.to(dev)

    def chain(x, cc, ucc):
        z, _ = smp.sample(S=DDIM_S, batch_size=B, shape=DDIM_SHAPE, conditioning=cc, verbose=False, x_T=x, eta=0.0,
                          unconditional_guidance_scale=DDIM_SCALE, unconditional_conditioning=ucc)
        return z

    def barrier():
        if n_gpus > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    chain(xT, c, uc)                                   # warm-up: sizes the arena, captures the step graph
    barrier()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(chains):
        z = chain(xT, c, uc)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = _lib.launch_count() - l0
    if outputs is not None:
        outputs["ddim_latent"] = z.cpu()
    # e2e: host tensors in, host latent out, through DDIMSampler.sample
    t0 = time.perf_counter()
    for _ in range(chains):
        z_h = chain(xT_h.to(dev, non_blocking=True), c_h.to(dev, non_blocking=True), uc_h.to(dev, non_blocking=True)).cpu()
    barrier()
    e2e_sec = (time.perf_counter() - t0) / chains
    if n_gpus > 1:
        tt = torch.tensor([ms, e2e_sec], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms, e2e_sec = float(tt[0].item()), float(tt[1].item())
    finite = bool(torch.isfinite(z).all().item())
    L = _lib.lib()
    L.agpt_unet_launches_per_step.restype = C.c_long
    lps = int(L.agpt_unet_launches_per_step(u._h))
    if keep is not None:
        keep["sampler"] = smp
    del smp, u
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    ms_chain = ms / chains
    clips = B * n_gpus
    value = clips / (ms_chain * 1e-3)
    ach = DDIM_TFLOP_PER_CLIP * B / (ms_chain * 1e-3)             # per GPU, algorithmic
    peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0)))
    ddim_traffic = None
    try:      # DRAM bytes of one 4-clip chain (100 steps) from the committed ncu launch list of the DDIM steps
        ddim_traffic = json.load(open(os.path.join(ROOT, "profiles", "ddim_traffic.json"))).get("dram_bytes_per_chain")
    except Exception:
        pass
    out = {"metric": DDIM_METRIC, "value": value, "unit": DDIM_UNIT, "n_gpus": n_gpus, "steps": chains, "warmup": 1,
           "ms_per_step": ms_chain, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic", "config": ddim_config(n_gpus),
           "value_per_gpu": value / n_gpus, "finite": finite,
           "e2e": {"value": clips / e2e_sec, "unit": DDIM_UNIT,
                   "h2d_bytes_per_step": int(xT_h.nbytes + c_h.nbytes + uc_h.nbytes), "d2h_bytes_per_step": int(z_h.nbytes),
                   "api": "DDIMSampler.sample(S=100, ...) on pinned host tensors -> .cpu() latent"},
           "gpu_launches": int(launches), "launches_per_ddim_step": lps,
           "roofline": {"kernel": "whole DDIM chain: tcconv5/6 tap-GEMMs + GroupNorm / LayerNorm / attention / update kernels",
                        "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                        "frac_issued": 3.0 * ach / peak, "algorithmic_tflop_per_clip": DDIM_TFLOP_PER_CLIP,
                        "peak_source": ("MEASURED_PEAKS.json bf16_tflops_sustained (a kernel timed inside a long step)"
                                        if peaks else "fallback 1.59 PFLOP/s dense bf16/fp16"),
                        "note": "achieved = 18.66 algorithmic TFLOP per clip x clips per GPU / chain time (all kernels of the "
                                "chain, not only the GEMMs); traffic = DRAM bytes of one chain (profiles/ddim_traffic.json)",
                        "traffic": ddim_traffic}}
    if want_cpu:
        r, sps, cores = cpu_ddim_rate(3)
        out["cpu_baseline"] = {"value": r, "unit": DDIM_UNIT, "cores": cores, "kind": "port",
                               "sample": f"B=1: 3 of the {DDIM_S} DDIM steps of oracle/ldm_ref.py (CFG pair per step) on {cores} threads; "
                                         f"clips/s = 1 / (s_per_step x {DDIM_S})"}
    return out


# ------------------------------------------------------------------------------------ GPU arm: mixed dispatch (C5)
def measure_mixed(dev, rank, n_gpus, vocoder, sampler):
    """BASELINE configs[4]: 64 concurrent prompts -- 32 TTS utterances (T ~ U{200..800} mel frames, seed 7, through
    HiFi-GAN) + 32 text-to-audio clips (DDIM-100 + CFG on the 4x10x78 latent -> AutoencoderKL.decode -> the 80x624 mel
    through the vocoder) -- assigned to the ranks by greedy LPT on the FLOP cost model (parallel.run_mixed), every
    rank serving its own jobs with no data-path collective; text-to-audio jobs of a rank run in micro-batches of 4
    clips.  Returns makespan, jobs/s and per-GPU busy fraction (all ranks get the same dict)."""
    from audiogpt_b200 import parallel, specs
    from audiogpt_b200.ldm.models.autoencoder import AutoencoderKL
    cfgv = specs.VAE_TXT2AUDIO
    vae = AutoencoderKL(ddconfig={k: v for k, v in cfgv.items() if k != "embed_dim"}, embed_dim=cfgv["embed_dim"])
    vae.load_state_dict(specs.synth_vae_decoder(cfgv, 5150), strict=False)
    vae = vae.eval().to(dev)
    rng = np.random.RandomState(7)
    jobs = [("tts", int(t)) for t in rng.randint(200, 801, 32)] + [("t2a", 624)] * 32
    done = {"tts": 0, "t2a": 0, "samples": 0}

    def run_group(kind, idxs):
        if kind == "tts":
            for i in idxs:
                mel = specs.synth_tensor((1, 80, jobs[i][1]), seed=1000 + i, scale=2.0, shift=-4.0).to(dev)
                done["samples"] += int(vocoder(mel).shape[-1])
                done["tts"] += 1
            return
        B = len(idxs)
        xT = torch.tensor(np.random.RandomState(55 + idxs[0]).randn(B, *DDIM_SHAPE), dtype=torch.float32).to(dev)
        c = specs.synth_tensor((B, 77, 1024), seed=2000 + idxs[0]).to(dev)
        uc = specs.synth_tensor((1, 77, 1024), seed=6).expand(B, -1, -1).contiguous().to(dev)
        z, _ = sampler.sample(S=DDIM_S, batch_size=B, shape=DDIM_SHAPE, conditioning=c, verbose=False, x_T=xT, eta=0.0,
                              unconditional_guidance_scale=DDIM_SCALE, unconditional_conditioning=uc)
        mel = vae.decode(z)[:, 0]                       # [B, 80, 624]
        done["samples"] += int(vocoder(mel.contiguous()).shape[-1]) * B
        done["t2a"] += B

    # warm-up of every engine shape class outside the clock (arena sizing, graph capture for the B=4 and tail batches)
    run_group("t2a", [32, 33, 34, 35])
    run_group("tts", [0])
    done.update(tts=0, t2a=0, samples=0)
    res = parallel.run_mixed(jobs, None, sync=lambda: torch.cuda.synchronize(dev), run_group=run_group,
                             group_size={"t2a": 4, "tts": 1})
    del vae
    torch.cuda.empty_cache()
    return {"workload": "BASELINE configs[4]: 32 TTS utterances (200..800 frames, HiFi-GAN V1) + 32 text-to-audio clips "
                        "(DDIM-100 CFG 1.5 -> AutoencoderKL.decode -> HiFi-GAN on the 80x624 mel), greedy LPT over the ranks, "
                        "text-to-audio in micro-batches of 4 clips per rank",
            "jobs": len(jobs), "makespan_s": res["makespan_s"], "jobs_per_s": res["jobs_per_s"],
            "busy_s": res["busy_s"], "busy_fraction": res["busy_fraction"],
            "model_load_tflop_per_rank": res["model_load_tflop"],
            "jobs_on_rank0": {"tts": done["tts"], "t2a": done["t2a"]}, "collectives_in_data_path": 0}


# ------------------------------------------------------------------------------------ GPU arm: HiFi-GAN
def run_ours(args):
    import ctypes as C
    from audiogpt_b200 import _lib, parallel, specs
    from audiogpt_b200.modules.hifigan.hifigan import HifiGanGenerator

    rank, world, local = parallel.init_distributed()
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    n_gpus = world
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    import torch.distributed as dist
    L = _lib.lib()
    L.agpt_fma_peak_tflops.restype = C.c_double
    peaks = load_peaks()

    def finish():
        if n_gpus > 1:
            dist.barrier()
            dist.destroy_process_group()

    outputs = {}
    if args.workload == "ddim":
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        d = measure_ddim(dev, rank, n_gpus, args.steps, peaks, want_cpu=(n_gpus == 1), outputs=outputs)
        if rank == 0:
            d["clocks"] = sampler.stop()
            if args.dump_outputs:
                dump_outputs(args.dump_outputs, outputs)
            print(json.dumps(d))
            sys.stdout.flush()
        finish()
        return

    h = specs.HIFIGAN_V1
    shapes = specs.hifigan_param_shapes(h)
    sd = specs.synth_hifigan(h, 1234) if rank == 0 else {k: torch.empty(s) for k, s in shapes.items()}
    sd = parallel.broadcast_state_dict(sd, src=0)          # the one weight broadcast (NCCL over NVLink)
    model = HifiGanGenerator(h)
    model.load_state_dict(sd, strict=True)
    model = model.eval().to(dev)
    mel_host = specs.synth_tensor((B_PER_GPU, 80, T_FRAMES), seed=100 + rank, scale=2.0, shift=-4.0)
    mel = mel_host.to(dev)
    frames_step = B_PER_GPU * T_FRAMES * n_gpus
    # finished waveforms -> every rank: asynchronous NCCL all-gather on NCCL's stream under the next step (default), or
    # AGPT_GATHER=p2p: copy engines over NVLink (parallel.P2PGather).  Measured on one 4-GPU box (profiles/r2w_*): no gather
    # 18.94 ms per step, NCCL 19.07, copy engines 19.86 -- N - 1 serial peer copies per rank stop paying past N = 2
    gather, gather_kind = None, None
    if n_gpus > 1:
        gsel = os.environ.get("AGPT_GATHER", "nccl")
        if gsel == "none":      # diagnostic: compute-only scaling (no waveform gather)
            gather, gather_kind = None, "none (diagnostic)"
        elif gsel == "p2p":
            try:
                gather, gather_kind = parallel.P2PGather((B_PER_GPU, 1, T_FRAMES * HOP), device=dev), "p2p_copy_engine"
            except RuntimeError as e:        # raised on every rank together (peer mapping unavailable): NCCL path instead
                print(f"[bench] {e}; using the NCCL gather", file=sys.stderr)
                gather, gather_kind = parallel.AsyncGather(), "nccl_async (p2p mapping failed)"
        else:
            gather, gather_kind = parallel.AsyncGather(), "nccl_async"

    def barrier():
        if n_gpus > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def step_device():
        wav = model(mel)
        if gather is not None:
            gather.submit(wav)       # finished waveforms -> every rank, on NCCL's stream, under the next step
        return wav

    for _ in range(args.warmup):
        step_device()
    if gather is not None:
        gather.drain()
    # the clock sampler forks nvidia-smi (tens of ms for a process of this size): start it BEFORE the barrier that aligns
    # the ranks -- started after it, rank 0 entered the timed loop late and every other rank's time (max over ranks)
    # included the wait for it at the final gather barrier (0.5 ms per step at N = 2, 6 ms at N = 4 with 10 steps)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        wav = step_device()
    if gather is not None:
        gather.drain()               # the compute stream waits for every outstanding gather: inside the timed region
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = _lib.launch_count() - l0
    outputs["hifigan_wav"] = wav.cpu()
    per_rank_ms = None
    if n_gpus > 1:
        allms = [torch.zeros(1, device=dev) for _ in range(n_gpus)]
        dist.all_gather(allms, torch.tensor([ms], device=dev))
        per_rank_ms = [float(t.item()) / args.steps for t in allms]
        ms = max(per_rank_ms) * args.steps
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = ms / args.steps
    value = frames_step / (ms_per_step * 1e-3)

    # ---- e2e: host buffers through the C-ABI (H2D + forward + D2H + sync inside the call)
    mel_np = mel_host.numpy()
    for _ in range(max(1, args.warmup // 2)):
        model.vocode_host(mel_np, device=dev)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        wav_np = model.vocode_host(mel_np, device=dev)
    barrier()
    e2e_sec = (time.perf_counter() - t0) / args.steps
    if n_gpus > 1:
        tt = torch.tensor([e2e_sec], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_sec = float(tt.item())
    e2e = {"value": frames_step / e2e_sec, "unit": UNIT,
           "h2d_bytes_per_step": int(mel_np.nbytes), "d2h_bytes_per_step": int(wav_np.nbytes),
           "api": "HifiGanGenerator.vocode_host -> agpt_hifigan_vocode_host (numpy in / numpy out)"}

    # ---- roofline of the dominant kernel, measured live with CUDA events around every launch (rank 0)
    roofline = None
    if rank == 0:
        fma_peak = float(L.agpt_fma_peak_tflops())
        _lib.check(L.agpt_profile_enable(1))
        model(mel)
        msv, flv, byv, lnv = (C.c_double * 4)(), (C.c_double * 4)(), (C.c_double * 4)(), (C.c_longlong * 4)()
        _lib.check(L.agpt_profile_collect(msv, flv, byv, lnv))
        _lib.check(L.agpt_profile_enable(0))
        tot_ms = sum(msv)
        ach_tf = sum(flv) / (tot_ms * 1e-3) / 1e12
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "tapconv_traffic.json"))).get("dram_bytes_per_launch")
        except Exception:
            pass
        variants = ["fma_BN128", "fma_BN64", "fma_BN32", "tcgen05_3xFP16"]
        tc_on = lnv[3] > 0
        per_variant = {variants[i]: {"launches": int(lnv[i]), "ms": msv[i],
                                     "tflops": (flv[i] / (msv[i] * 1e-3) / 1e12) if msv[i] > 0 else None,
                                     "gbs": (byv[i] / (msv[i] * 1e-3) / 1e9) if msv[i] > 0 else None}
                       for i in range(4) if lnv[i] > 0}
        hbm = {"bound": "hbm", "achieved": sum(byv) / (tot_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
               "frac": sum(byv) / (tot_ms * 1e-3) / 1e9 / hbm_peak,
               "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6.65 TB/s",
               "note": "per-launch algorithmic bytes (in+out+residual+weights of every conv launch); the path is compute-bound "
                       "(AI ~ 10^3 FLOP/B, SURVEY.md 8d) so this fraction is small by construction"}
        if tc_on:
            f16_peak = float(peaks.get("bf16_tflops", 1590.0))
            roofline = {
                "kernel": "tcconv6_kernel<BN,NI> / tcconv5_kernel<BN,NWK> (tcgen05 tap-GEMM, 3 x fp16 hi/lo products; "
                          "all contractions of the generator)",
                "bound": "tensor", "achieved": ach_tf, "peak": f16_peak, "unit": "TFLOP/s",
                "frac": ach_tf / f16_peak, "frac_issued": 3.0 * ach_tf / f16_peak,
                "achieved_issued_tflops": 3.0 * ach_tf,
                "peak_source": ("MEASURED_PEAKS.json bf16_tflops (burst: kernels timed one by one); kind::f16 issues at the bf16 rate"
                                if peaks else "fallback 1.59 PFLOP/s dense bf16/fp16"),
                "note": "achieved / frac are on ALGORITHMIC FLOPs (SURVEY.md 8d: 0.614 GFLOP per mel frame, zero-padded polyphase "
                        "taps not counted); the tensor pipe issues 3 fp16 products per fp32-grade MAC (frac_issued)",
                "fp32_fma_peak_tflops_measured": fma_peak,
                "algorithmic_vs_fp32_fma_peak": ach_tf / fma_peak if fma_peak > 0 else None,
                "share_of_step": tot_ms / ms_per_step if n_gpus == 1 else None,
                "per_variant": per_variant, "hbm": hbm, "traffic": traffic,
            }
        else:
            roofline = {
                "kernel": "tapconv_kernel<BN> (fp32 FMA; all contractions of the generator)",
                "bound": "fma_fp32", "achieved": ach_tf, "peak": fma_peak, "unit": "TFLOP/s",
                "frac": ach_tf / fma_peak if fma_peak > 0 else None,
                "peak_source": "fp32 FFMA saturation probe run in this process (agpt_fma_peak_tflops)",
                "share_of_step": tot_ms / ms_per_step if n_gpus == 1 else None,
                "per_variant": per_variant, "hbm": hbm, "traffic": traffic,
            }
    # ---- the other half of the metric: DDIM-100 clips/s on the C4 shard (all ranks), then the mixed dispatch (C5)
    ddim, mixed, keep = None, None, {}
    if not args.no_ddim:
        try:
            ddim = measure_ddim(dev, rank, n_gpus, args.ddim_chains, peaks, want_cpu=False, keep=keep, outputs=outputs)
        except Exception as ex:
            if n_gpus > 1:
                raise
            ddim = {"error": repr(ex)}
        if keep.get("sampler") is not None and not args.no_mixed:
            try:
                mixed = measure_mixed(dev, rank, n_gpus, model, keep["sampler"])
            except Exception as ex:
                if n_gpus > 1:
                    raise
                mixed = {"error": repr(ex)}
    keep.clear()
    del model
    torch.cuda.empty_cache()
    if rank != 0:
        finish()
        return

    # ---- CPU baseline on this box's host cores (bounded sample)
    if n_gpus == 1:
        cb_rate, cb_sec, cores = cpu_vocode_rate(3, 1, 2, T_FRAMES)
        cpu_baseline = {"value": cb_rate, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": f"2 of {B_PER_GPU} utterances x {T_FRAMES} frames in one forward call, 1 warm-up + 3 timed passes of "
                                  f"oracle/hifigan_ref.py on {cores} threads (best of a thread-count calibration; "
                                  f"box has {os.cpu_count()} logical CPUs); {_ALLOC_NOTE}"}
        if ddim and "error" not in ddim:
            r, sps, dcores = cpu_ddim_rate(3)
            ddim["cpu_baseline"] = {"value": r, "unit": DDIM_UNIT, "cores": dcores, "kind": "port",
                                    "sample": f"B=1: 3 of the {DDIM_S} DDIM steps of oracle/ldm_ref.py (CFG pair per step) on "
                                              f"{dcores} threads; clips/s = 1 / (s_per_step x {DDIM_S})"}
    else:
        cpu_baseline = None   # timed at N=1 only (torchrun pins OMP_NUM_THREADS=1 per rank)

    extra = {}
    if not args.no_extra and n_gpus == 1:
        try:
            extra = extra_metrics(dev)
        except Exception as ex:  # extras must never take the headline down
            extra = {"error": repr(ex)}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": base_config(n_gpus),
            "x_realtime": value * HOP / SR, "x_realtime_per_gpu": value * HOP / SR / n_gpus,
            "tflops_fp32": 0.614e9 * value / 1e12,
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
            "roofline": roofline, "cpu_baseline": cpu_baseline, "ddim": ddim, "mixed_dispatch": mixed, "extra": extra,
            "waveform_gather": gather_kind, "ms_per_step_by_rank": per_rank_ms}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line))
    sys.stdout.flush()
    finish()


def extra_metrics(dev):
    """Secondary measurements, each one complete run: the C3 DiffSinger chain (16 utt x 400 frames, 100 ancestral
    p_sample steps on the device loop) -> utterances/s; BigVGAN base (the vocoder Make-An-Audio dispatches)."""
    import ctypes as C
    from audiogpt_b200 import _lib, specs
    from audiogpt_b200.modules.diff import shallow_diffusion_tts as sdt
    from audiogpt_b200.modules.diff.net import DiffNet
    from audiogpt_b200.utils.hparams import set_hparams_from_dict
    out = {}
    # --- C3
    cfgd = specs.DIFFNET_BASE
    set_hparams_from_dict(dict(cfgd, keep_bins=80, schedule_type="linear", max_beta=0.06))
    net = DiffNet(80)
    net.load_state_dict(specs.synth_diffnet(cfgd, 2025), strict=True)
    gd = sdt.GaussianDiffusion(None, 80, net, timesteps=100, K_step=100, loss_type="l1",
                               betas=sdt.linear_beta_schedule(100, 0.06), spec_min=specs.SPEC_MIN,
                               spec_max=specs.SPEC_MAX).eval().to(dev)
    Bc, Tc = 16, 400
    x = specs.synth_tensor((Bc, 1, 80, Tc), seed=2).to(dev)
    cond = specs.synth_tensor((Bc, 256, Tc), seed=3).to(dev)
    gd.sample(cond, x_start=x)                         # warm-up (captures the step graph)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    gd.sample(cond, x_start=x)                         # includes drawing the 100 noise tensors, as the reference's loop does
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    out["diffsinger_c3_utt_per_s"] = Bc / dt
    out["diffsinger_c3_seconds_16utt_100steps"] = dt
    out["diffsinger_c3_tflops_algorithmic"] = 26.44e6 * Bc * Tc * 100 / dt / 1e12
    Lb = _lib.lib()
    Lb.agpt_diffnet_launches_per_step.restype = C.c_long
    out["diffsinger_c3_launches_per_step"] = int(Lb.agpt_diffnet_launches_per_step(net._h))
    del net, gd
    torch.cuda.empty_cache()
    # --- AutoencoderKL.decode ("next" row 8f-1): 4 latents 4x10x78 -> 4 mel images 1x80x624 (392.9 GFLOP per clip)
    from audiogpt_b200.ldm.models.autoencoder import AutoencoderKL
    cfgv = specs.VAE_TXT2AUDIO
    vae = AutoencoderKL(ddconfig={k: v for k, v in cfgv.items() if k != "embed_dim"}, embed_dim=cfgv["embed_dim"])
    vae.load_state_dict(specs.synth_vae_decoder(cfgv, 5150), strict=False)
    vae = vae.eval().to(dev)
    zz = specs.synth_tensor((4, 4, 10, 78), seed=3).to(dev)
    for _ in range(2):
        vae.decode(zz)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        ym = vae.decode(zz)
    e1.record()
    torch.cuda.synchronize(dev)
    msv = e0.elapsed_time(e1) / 3
    out["vae_decode_ms_4clips"] = msv
    out["vae_decode_clips_per_s"] = 4 / (msv * 1e-3)
    out["vae_decode_tflops_algorithmic"] = 0.3929 * 4 / (msv * 1e-3)
    out["vae_decode_finite"] = bool(torch.isfinite(ym).all().item())
    del vae
    torch.cuda.empty_cache()
    # --- BigVGAN ("next" row 8f-2: the vocoder Make-An-Audio actually dispatches), base 22 kHz / 80-band topology
    from audiogpt_b200.vocoder.bigvgan.models import BigVGAN
    hb = specs.BIGVGAN_BASE
    bv = BigVGAN(hb)
    bv.load_state_dict(specs.synth_bigvgan(hb, 4321), strict=True)
    bv = bv.eval().to(dev)
    Bb, Tb = 8, 400
    melb = specs.synth_tensor((Bb, 80, Tb), seed=9, scale=2.0, shift=-4.0).to(dev)
    for _ in range(2):
        bv(melb)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        wb = bv(melb)
    e1.record()
    torch.cuda.synchronize(dev)
    msb = e0.elapsed_time(e1) / 3
    out["bigvgan_base_frames_per_s"] = Bb * Tb / (msb * 1e-3)
    out["bigvgan_base_ms_8x400"] = msb
    out["bigvgan_base_finite"] = bool(torch.isfinite(wb).all().item())
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="hifigan", choices=["hifigan", "ddim"],
                    help="hifigan (default): the contract line, with the DDIM C4 measurement under 'ddim'; "
                         "ddim: the C4 DDIM-100 line alone (steps = timed chains)")
    ap.add_argument("--ddim-chains", type=int, default=2, help="timed DDIM-100 chains of the 'ddim' object (after 1 warm-up chain)")
    ap.add_argument("--no-ddim", action="store_true", help="skip the DDIM C4 measurement")
    ap.add_argument("--no-mixed", action="store_true", help="skip the mixed-dispatch (BASELINE configs[4]) measurement")
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary DiffSinger / BigVGAN measurements")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32, GPU arm only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (audiogpt_b200 has no CPU fallback)")
        run_ours(args)


if __name__ == "__main__":
    main()

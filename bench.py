#!/usr/bin/env python
"""bench.py — SUPIR EDM sampling hot path on B200: megapixels/sec and ms/EDM-step.

Default workload = BASELINE.json configs[2] ("cfg3", the configuration the metric is quoted on; it fits one GPU): one
1024x1024 image restored at upscale 4 -> 4096x4096 output (16.78 MP), latent 512x512, `TiledRestoreEDMSampler(tile 128,
stride 64)` = 49 windows per step (the gradio_demo_tiled.py reading of the config, the one that shards over GPUs),
cond+uncond CFG pair, s_churn 5, s_noise 1.01, linear CFG 1.0 -> 4.0, tiled VAE (encoder tile 1024 px, decoder tile 128
latent). `--config cfg2 | cfg4 | cfg5` select the other BASELINE configurations (WORKLOADS below). Synthetic input,
random-init weights of the exact SUPIR-v0 / SDXL-base / SDXL-VAE architecture.

Everything runs through the engine API a user calls (supir_b200.model.SUPIRModel: encode_first_stage_with_denoise /
decode_first_stage / encode_first_stage, the sampler it instantiates from the YAML-shaped config, batchify_sample).

A "step" is ONE sampler step: every window x (control net + UNet) on the CFG pair, the step arithmetic, the window blend
(and, for N > 1, the all-gather of the network outputs). `ms_per_step` is its device time over EXACTLY K steps. `value`
(megapixels/sec) is output MP / (steps_of_the_config * ms_per_step + the VAE passes (2 encodes + 2 decodes) timed in the
same run). `e2e` repeats both with host buffers in the loop (pinned host -> device copy of the step's latent and
device -> host read-back of the result every step; image upload + decoded image download around the VAE). `full_run` is ONE
real `SUPIRModel.batchify_sample` call of the whole configuration (image on the host in, image on the host out), wall-clock
— the same quantity measured without any arithmetic. N > 1 shards the windows / tiles of the SAME image over ranks (strong
scaling; cfg2 / cfg5 do not shard: N independent replicas, weak scaling).

`--impl reference` times the CPU oracle (the reference algorithm restated in fp32 PyTorch) on the host cores: a "step" there
is one bounded sample of the workload — one denoiser call (control + UNet, CFG pair) on ONE 128x128 latent window, 1/49 of an
EDM step of cfg3 — and `value` is the whole-job throughput that sample time implies (x windows x steps, plus the VAE tiles).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

UNET_CFG = dict(adm_in_channels=2816, num_classes="sequential", use_checkpoint=True, in_channels=4, out_channels=4,
                model_channels=320, attention_resolutions=[4, 2], num_res_blocks=2, channel_mult=[1, 2, 4],
                num_head_channels=64, use_spatial_transformer=True, use_linear_in_transformer=True,
                transformer_depth=[1, 2, 10], context_dim=2048, spatial_transformer_attn_type="softmax-xformers", legacy=False)
VAE_CFG = dict(attn_type="vanilla-xformers", double_z=True, z_channels=4, resolution=256, in_channels=3, out_ch=3, ch=128,
               ch_mult=[1, 2, 4, 4], num_res_blocks=2, attn_resolutions=[], dropout=0.0)
DISC = {"target": "sgm.modules.diffusionmodules.discretizer.LegacyDDPMDiscretization"}
# algorithmic FLOP of one denoiser call (control + UNet, CFG pair) by latent side: SURVEY.md §8(d), BASELINE.md §3
FLOP_BY_LATENT = {64: 4.766e12, 128: 20.292e12, 256: 107.887e12, 512: 866.071e12}
FLOP_WINDOW = FLOP_BY_LATENT[128]
# VAE conv + norm work per output/input megapixel and the mid-block attention term (SURVEY.md §8d)
VAE_ENC_FLOP_PER_MP, VAE_DEC_FLOP_PER_MP = 4.33e12, 9.92e12

# BASELINE.json configs[1..4]. `windows` is filled in from the sampler's own window list at run time.
WORKLOADS = {
    "cfg3": dict(in_px=1024, upscale=4, sampler="TiledRestoreEDMSampler", tile=128, stride=64, steps=50, enc_tile=1024, dec_tile=128,
                 shards=True, images_per_gpu=1,
                 desc="1024x1024->4096x4096 (16.78 MP), 50 EDM steps, TiledRestoreEDMSampler 128/64 = 49 windows, CFG pair, "
                      "tiled VAE enc 1024 px / dec 128 latent"),
    "cfg2": dict(in_px=1024, upscale=2, sampler="RestoreEDMSampler", tile=None, stride=None, steps=50, enc_tile=None, dec_tile=None,
                 shards=False, images_per_gpu=1,
                 desc="1024x1024 input, upscale 2 -> 2048x2048 (4.19 MP), 50 EDM steps, untiled RestoreEDMSampler on the 256x256 "
                      "latent (16 384-token self-attention), CFG pair, untiled VAE; one image per GPU (replicas only)"),
    "cfg2pair": dict(in_px=1024, upscale=2, sampler="RestoreEDMSampler", tile=None, stride=None, steps=50, enc_tile=None, dec_tile=None,
                     shards=True, images_per_gpu=1,
                     desc="cfg2 in latency mode: ONE 1024 -> 2048x2048 image on TWO GPUs, the unconditional / conditional CFG branch "
                          "of every untiled step on its own GPU, one all-gather of the network outputs per step (VAE replicated)"),
    "cfg4": dict(in_px=2048, upscale=4, sampler="TiledRestoreEDMSampler", tile=128, stride=64, steps=50, enc_tile=512, dec_tile=64,
                 shards=True, images_per_gpu=1,
                 desc="2048x2048->8192x8192 (67.1 MP), 50 EDM steps, TiledRestoreEDMSampler 128/64 = 225 windows, CFG pair, tiled VAE "
                      "at the reference defaults (enc 512 px / dec 64 latent = 256 tiles each), windows and tiles sharded over ranks"),
    "cfg5": dict(in_px=1024, upscale=2, sampler="RestoreDPMPP2MSampler", tile=None, stride=None, steps=4, enc_tile=None, dec_tile=None,
                 shards=False, images_per_gpu=1,
                 desc="Juggernaut-lightning path: RestoreDPMPP2MSampler, 4 steps, 1024 -> 2048x2048 (4.19 MP) per image, CFG pair, "
                      "untiled VAE; one image per GPU (throughput mode, replicas only)"),
}


def flop_denoiser(side):
    if side in FLOP_BY_LATENT:
        return FLOP_BY_LATENT[side]
    hw = side * side
    return 1.1e9 * hw + 0.1416e12 * (hw / 4096.0) ** 2


def workload_geometry(w):
    out_px = w["in_px"] * w["upscale"]
    latent = out_px // 8
    if w["tile"]:
        from supir_b200.sampling import _sliding_windows
        windows = len(_sliding_windows(latent, latent, w["tile"], w["stride"]))
        step_flop = windows * flop_denoiser(w["tile"])
    else:
        windows = 1
        step_flop = flop_denoiser(latent)
    return out_px, latent, windows, step_flop


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p["bf16_tflops_sustained"], p["bf16_tflops"], p["hbm_gbs"], "measured"
    except Exception:
        return 1400.0, 1590.0, 6650.0, "fallback"


def load_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed ncu capture."""
    for name in ("r02_gemm_traffic.json", "r01_gemm_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                return json.load(f)["dram_bytes_per_launch_mean"], name
        except Exception:
            continue
    return None, None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index, self.proc, self.lines, self.i0 = index, None, [], 0

    def mark(self):
        """Start of the timed region: samples read from here on are the ones reported. The process is started before the
        warm-up steps because nvidia-smi needs up to a second to emit its first line on a multi-GPU box."""
        self.i0 = len(self.lines)

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        window = "timed region"
        lines = self.lines[self.i0:]
        if not any(len(ln.split(",")) >= 7 for ln in lines):
            lines, window = self.lines[-8:], "warm-up + timed steps (same load; no sample fell inside the short timed region)"
        sm, mx, reasons = [], None, set()
        for ln in lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm),
                "window": window}


# ------------------------------------------------------------------------------------------------------------------
# CPU oracle timing (cpu_baseline leg and --impl reference)
# ------------------------------------------------------------------------------------------------------------------
def oracle_state_dict(fast=False, depth=None):
    """Random fp32 weights with the full SUPIR-v0 shapes, keyed like the reference checkpoint (model.* prefix dropped).
    `fast` (timing legs only): every tensor is cut from one 16 M-element normal block instead of 3.87 G fresh draws — dense
    fp32 GEMM time does not depend on the values, and the single-threaded generator would otherwise cost over a minute."""
    from supir_b200 import nets
    cfg = UNET_CFG if depth is None else dict(UNET_CFG, transformer_depth=depth)      # `depth`: tests/test_bench_contract.py only
    with torch.device("meta"):
        unet = nets.LightGLVUNet(mode="XL-base", project_type="ZeroSFT", project_channel_scale=2, **cfg)
        ctrl = nets.GLVControl(input_upscale=1, **cfg)
    sd = {}
    g = torch.Generator().manual_seed(0)
    block = torch.randn(1 << 24, generator=g) if fast else None
    for prefix, m in (("diffusion_model.", unet), ("control_model.", ctrl)):
        for k, v in m.state_dict().items():
            if k.endswith("weight") and v.dim() >= 2:
                fan_in = int(np.prod(v.shape[1:]))
                if fast:
                    n, bn = v.numel(), block.numel()
                    t = torch.empty(n, dtype=torch.float32)
                    scaled = block * (1.0 / fan_in ** 0.5)
                    reps = n // bn
                    if reps:
                        t[:reps * bn].view(reps, bn).copy_(scaled.expand(reps, bn))
                    t[reps * bn:].copy_(scaled[:n - reps * bn])
                    t = t.view(v.shape)
                else:
                    t = torch.empty(v.shape, dtype=torch.float32).normal_(0, 1.0 / fan_in ** 0.5, generator=g)
            elif k.endswith("weight"):
                t = torch.ones(v.shape, dtype=torch.float32)
            else:
                t = torch.zeros(v.shape, dtype=torch.float32)
            sd[prefix + k] = t
    return sd


def oracle_vae_state_dict():
    from supir_b200 import vae
    with torch.device("meta"):
        ae = vae.AutoencoderKLInferenceWrapper(embed_dim=4, ddconfig=VAE_CFG, lossconfig={"target": "torch.nn.Identity"})
    sd = {}
    g = torch.Generator().manual_seed(1)
    for k, v in ae.state_dict().items():
        t = torch.empty(v.shape, dtype=torch.float32)
        if k.endswith("weight") and v.dim() >= 2:
            t.normal_(0, 1.0 / int(np.prod(v.shape[1:])) ** 0.5, generator=g)
        elif k.endswith("weight"):
            t.fill_(1.0)
        else:
            t.zero_()
        sd[k] = t
    return sd


def time_oracle_window(sd, side, repeats):
    """Seconds per denoiser call (control + UNet on the CFG pair, B=2) on one side x side latent window, fp32 CPU."""
    from oracle import unet as ounet
    x = torch.randn(2, 4, side, side)
    cond = {"control": torch.randn(2, 4, side, side), "crossattn": torch.randn(2, 77, 2048), "vector": torch.randn(2, 2816)}
    t = torch.tensor([500, 500])
    times = []
    with torch.no_grad():
        for _ in range(repeats):
            t0 = time.perf_counter()
            ounet.control_wrapper_forward(sd, x, t, cond, 1.0)
            times.append(time.perf_counter() - t0)
    return times


def probe_oracle_window(sd, budget_s, want_calls):
    """Seconds of ONE oracle denoiser call on the 128x128 latent window of the tiled sampler.

    The 128-latent window is timed DIRECTLY whenever one call fits what is left of `budget_s` (as many of `want_calls` calls
    as fit, at least one); its cost is first predicted from single calls at 32 and 64 by the two-point fit
    t = a + b * FLOP(side) (a = the size-independent cost of streaming 15.5 GB of fp32 weights). Only if even one call does
    not fit is that fit reported instead — never a single small window scaled by FLOPs.
    Returns (seconds per 128-window call, {side: [seconds...]}, 'measured' | 'two-point fit')."""
    t_begin = time.perf_counter()
    time_oracle_window(sd, 16, 1)        # warm-up: first touch of the weights, oneDNN primitive creation
    meas = {32: time_oracle_window(sd, 32, 1), 64: time_oracle_window(sd, 64, 1)}
    m32, m64 = meas[32][0], meas[64][0]
    b = max((m64 - m32) / (flop_denoiser(64) - flop_denoiser(32)), 0.0)
    a = max(m64 - b * flop_denoiser(64), 0.0)
    predicted = a + b * FLOP_WINDOW
    left = budget_s - (time.perf_counter() - t_begin)
    n = int(min(want_calls, left // max(predicted * 1.1, 1e-3)))
    if n < 1:
        return predicted, meas, "two-point fit"
    meas[128] = time_oracle_window(sd, 128, n)
    return float(np.mean(meas[128])), meas, "measured"


def time_oracle_vae(budget_s, enc_tile_px, dec_tile_latent):
    """Seconds of the oracle VAE on ONE padded encoder tile and ONE padded decoder tile of the workload's tiling. If the full
    tile does not fit the budget a half-size tile is timed and scaled by pixel count (conv-bound; the quadratic mid-block
    attention term is then under-counted, which flatters the CPU)."""
    from oracle import vae as ovae
    sd = oracle_vae_state_dict()
    out, notes = {}, []
    for name, full, is_dec, flop_mp in (("enc", enc_tile_px, False, VAE_ENC_FLOP_PER_MP), ("dec", dec_tile_latent, True, VAE_DEC_FLOP_PER_MP)):
        mp_full = (full * (8 if is_dec else 1)) ** 2 / 1e6
        est = flop_mp * mp_full / 0.7e12          # ~0.7 TFLOP/s fp32 convs on a 64-core host: only used to pick the sample size
        side = full if est <= budget_s / 2 else max(full // 2 // 8 * 8, 64 if not is_dec else 16)
        x = torch.randn(1, 4 if is_dec else 3, side, side)
        with torch.no_grad():
            t0 = time.perf_counter()
            ovae.forward(sd, "decoder." if is_dec else "encoder.", x, is_dec)
            t = time.perf_counter() - t0
        out[name] = t * (full / side) ** 2
        notes.append(f"{name} tile {full}{' latent' if is_dec else ' px'}: {t:.2f} s at side {side}" + ("" if side == full else " (scaled by pixels)"))
    return out["enc"], out["dec"], "; ".join(notes)


def cpu_model(wname, sec_window, enc_tile_s, dec_tile_s):
    """Whole-job seconds of the CPU reference path for workload `wname` from the measured samples."""
    from supir_b200 import vae
    w = WORKLOADS[wname]
    out_px, latent, windows, step_flop = workload_geometry(w)
    per_step = sec_window * step_flop / FLOP_WINDOW
    sampling_s = per_step * w["steps"]
    if w["enc_tile"]:
        n_enc = len(vae.split_tiles(out_px, out_px, w["enc_tile"], False)[0])
        n_dec = len(vae.split_tiles(latent, latent, w["dec_tile"], True)[0])
        ref_enc, ref_dec = w["enc_tile"] + 64, w["dec_tile"] + 22
    else:
        n_enc = n_dec = 1
        ref_enc, ref_dec = out_px, latent
    # the sampled tiles are cfg3's (1088 px / 150 latent); other tilings scale by pixel count
    enc_s = enc_tile_s * (ref_enc / 1088.0) ** 2 * n_enc
    dec_s = dec_tile_s * (ref_dec / 150.0) ** 2 * n_dec
    vae_s = 2 * enc_s + 2 * dec_s
    return sampling_s + vae_s, per_step, vae_s


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = min(os.cpu_count() or 1, int(os.environ.get("SUPIR_BENCH_CPU_THREADS", "64")))
    torch.set_num_threads(cores)
    w = WORKLOADS[args.config]
    out_px, latent, windows, step_flop = workload_geometry(w)
    mp = out_px * out_px / 1e6
    total_budget = float(os.environ.get("SUPIR_BENCH_REF_BUDGET_S", "170"))
    t0 = time.perf_counter()
    # SUPIR_BENCH_REF_SHALLOW=1 (the CPU contract test only; never set by the driver): depth-1 transformers, 1 B instead of 3.9 B
    # parameters, so the line's SHAPE can be checked in seconds on a small host — its value is then NOT a benchmark number
    shallow = os.environ.get("SUPIR_BENCH_REF_SHALLOW", "0") == "1"
    sd = oracle_state_dict(fast=True, depth=[1, 1, 1] if shallow else None)
    build_s = time.perf_counter() - t0
    sec_window, meas, how = probe_oracle_window(sd, total_budget * 0.75, max(args.steps, 1))
    del sd
    enc_s, dec_s, vae_note = time_oracle_vae(total_budget * 0.25, 1088, 150)
    total_s, per_step_s, vae_s = cpu_model(args.config, sec_window, enc_s, dec_s)
    n_timed = len(meas.get(128, []))
    sample = (f"oracle (fp32 PyTorch restatement of the reference, {cores} threads): control+UNet on ONE 128x128-latent window, CFG pair: "
              f"{how} {sec_window:.2f} s/call" + (f" over {n_timed} timed call(s) of the {args.steps} asked (budget {total_budget:.0f} s)" if n_timed else
                                                 f" (one call would not fit the {total_budget:.0f} s budget)") +
              f"; probes 32: {meas[32][0]:.2f} s, 64: {meas[64][0]:.2f} s; VAE: {vae_note}; job = {windows} window(s) x {w['steps']} steps "
              f"(by denoiser FLOPs for non-128 latents) + 2 encodes + 2 decodes")
    value = mp / total_s
    print(json.dumps({
        "impl": "reference", "metric": "megapixels_per_sec", "value": value, "unit": "MP/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec_window * 1e3, "higher_is_better": True,
        "scaling": "strong" if w["shards"] else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.config}: " + w["desc"] + " — CPU reference arm, extrapolated from a bounded sample",
                   "step_definition": "one bounded sample = one denoiser call on one 128x128 latent window (1/%d of a sampler step of this config)" % max(int(round(step_flop / FLOP_WINDOW)), 1),
                   "steps_timed": n_timed, "window_seconds": sec_window, "window_time_source": how,
                   "sampler_step_seconds_extrapolated": per_step_s, "vae_seconds_extrapolated": vae_s, "job_seconds_extrapolated": total_s,
                   "weights_build_seconds": build_s, **({"contract_check_only": "SUPIR_BENCH_REF_SHALLOW=1: depth-1 networks, not a benchmark number"} if shallow else {})},
        "cpu_baseline": {"value": value, "unit": "MP/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------------
def engine_config(w, tile_batch):
    sampler_params = {"num_steps": w["steps"], "restore_cfg": -1.0, "s_churn": 5, "s_noise": 1.01, "discretization_config": DISC,
                      "guider_config": {"target": "sgm.modules.diffusionmodules.guiders.LinearCFG", "params": {"scale": 1.0, "scale_min": 4.0}}}
    if w["tile"]:
        sampler_params.update(tile_size=w["tile"], tile_stride=w["stride"], tile_batch=tile_batch)
    if w["sampler"] == "RestoreDPMPP2MSampler":
        sampler_params.update(eta=1.0)
        sampler_params.pop("s_churn")
    return dict(
        control_stage_config={"target": "SUPIR.modules.SUPIR_v0.GLVControl", "params": dict(UNET_CFG, input_upscale=1)},
        network_config={"target": "SUPIR.modules.SUPIR_v0.LightGLVUNet",
                        "params": dict(UNET_CFG, mode="XL-base", project_type="ZeroSFT", project_channel_scale=2)},
        network_wrapper="sgm.modules.diffusionmodules.wrappers.ControlWrapper",
        denoiser_config={"target": "sgm.modules.diffusionmodules.denoiser.DiscreteDenoiserWithControl",
                         "params": {"num_idx": 1000, "weighting_config": {"target": "sgm.modules.diffusionmodules.denoiser_weighting.EpsWeighting"},
                                    "scaling_config": {"target": "sgm.modules.diffusionmodules.denoiser_scaling.EpsScaling"},
                                    "discretization_config": DISC}},
        first_stage_config={"target": "sgm.models.autoencoder.AutoencoderKLInferenceWrapper",
                            "params": {"embed_dim": 4, "ddconfig": VAE_CFG, "lossconfig": {"target": "torch.nn.Identity"}}},
        sampler_config={"target": "sgm.modules.diffusionmodules.sampling." + w["sampler"], "params": sampler_params},
        ae_dtype="bf16", diffusion_dtype="bf16", scale_factor=0.13025)


def build_engine(w, device, world):
    """supir_b200.model.SUPIRModel (the reference's SUPIRModel surface) with random bf16 weights of the real architecture."""
    from supir_b200 import model as smodel
    tile_batch = int(os.environ.get("SUPIR_BENCH_TILE_BATCH", "49"))
    with torch.device(device):
        m = smodel.SUPIRModel(**engine_config(w, tile_batch))
    m.model.diffusion_model.to(torch.bfloat16)
    m.model.control_model.to(torch.bfloat16)
    if w["enc_tile"]:
        m.init_tile_vae(encoder_tile_size=w["enc_tile"], decoder_tile_size=w["dec_tile"])
    if world > 1 and w["shards"]:
        m.enable_tile_sharding()
    m.model.pack()
    return m


def profile_dominant_kernel(net, device):
    """Live roofline of the dominant kernel (the tcgen05 GEMM / implicit-GEMM conv): one eager denoiser call with a
    CUDA-event pair (current stream) around every GEMM-class launch of the plan the timed steps replayed; achieved = sum of
    the launches' algorithmic FLOPs / sum of their durations."""
    from supir_b200 import ops
    rec = []
    orig_gemm, orig_conv = ops.gemm, ops.conv3x3

    def gemm(a, w, out, **kw):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = orig_gemm(a, w, out, **kw)
        e1.record()
        rec.append((2.0 * a.shape[0] * w.shape[0] * a.shape[1], e0, e1, ("gemm", a.shape[0], w.shape[0], a.shape[1], kw.get("act", 0))))
        return r

    def conv(x, B, H, W, wp, out, **kw):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = orig_conv(x, B, H, W, wp, out, **kw)
        e1.record()
        rec.append((2.0 * x.shape[0] * wp.shape[0] * wp.shape[1], e0, e1, ("conv3x3", x.shape[0], wp.shape[0], wp.shape[1], kw.get("act", 0))))
        return r

    if not net._plans:
        return None
    plan = net._plans[max(net._plans, key=lambda k: k[0] * k[1] * k[2])]
    plan._run()
    torch.cuda.synchronize()
    ops.gemm, ops.conv3x3 = gemm, conv
    try:
        plan._run()
        torch.cuda.synchronize()
    finally:
        ops.gemm, ops.conv3x3 = orig_gemm, orig_conv
    flops = sum(r[0] for r in rec)
    ms = sum(r[1].elapsed_time(r[2]) for r in rec)
    dump = os.environ.get("SUPIR_BENCH_DUMP_SHAPES")
    if dump:
        agg = {}
        for f, e0, e1, key in rec:
            a = agg.setdefault(key, [0, 0.0, 0.0])
            a[0] += 1
            a[1] += e0.elapsed_time(e1)
            a[2] += f
        rows = sorted(({"op": k[0], "M": k[1], "N": k[2], "K": k[3], "act": k[4], "count": v[0], "ms": round(v[1], 3),
                        "tflops": round(v[2] / (v[1] * 1e-3) / 1e12, 1)} for k, v in agg.items()), key=lambda r: -r["ms"])
        with open(dump, "w") as f:
            json.dump({"total_ms": ms, "total_tflop": flops / 1e12, "rows": rows, "order": [list(r[3]) for r in rec]}, f, indent=0)
    return flops, ms, len(rec), plan.key


def run_supir(args):
    import torch.distributed as dist
    from supir_b200 import _native, sampling
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = f"cuda:{local}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(device))
    w = WORKLOADS[args.config]
    out_px, latent, windows, step_flop = workload_geometry(w)
    shards = w["shards"] and world > 1
    images = 1 if w["shards"] else world                      # replicas: one image per rank
    megapixels = out_px * out_px / 1e6 * images
    # sharded: same seed on every rank (identical noise draws, see sampling.py); replicas: a different image per rank
    torch.manual_seed(1234 if w["shards"] else 1234 + rank)
    m = build_engine(w, device, world)
    net = m.model
    sust, burst, hbm, peak_kind = peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- inputs: pinned host buffers (synthetic LQ image already resized to the output resolution, like PIL2Tensor) ----
    img_host = torch.empty(1, 3, out_px, out_px, dtype=torch.float32).uniform_(-1, 1).pin_memory()
    out_host = torch.empty(1, 3, out_px, out_px, dtype=torch.float32).pin_memory()
    c = {"crossattn": torch.randn(1, 77, 2048, device=device), "vector": torch.randn(1, 2816, device=device)}
    uc = {"crossattn": torch.randn(1, 77, 2048, device=device), "vector": torch.randn(1, 2816, device=device)}
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

    # ---- VAE passes before sampling (SUPIR_model.py:117-119), timed; e2e includes the image upload ----
    skip_vae = os.environ.get("SUPIR_BENCH_SKIP_VAE", "0") == "1"     # profiling aid only: invalid as a benchmark number
    if not skip_vae:
        # untimed warm-up of the VAE passes (kernel module loads, scratch pools), the counterpart of the W warm-up steps
        for _ in range(min(args.warmup, 1)):
            _w = img_host.to(device)
            _wz = m.encode_first_stage_with_denoise(_w, use_sample=False)
            _wx = m.decode_first_stage(_wz)
            _wz2 = m.encode_first_stage(_wx)          # the third network of the pre-sampling passes has its own scratch pool
            del _w, _wz, _wx, _wz2
    barrier()
    e0, e1, e2 = ev(), ev(), ev()
    e0.record()
    img = img_host.to(device, non_blocking=True)
    e1.record()
    if skip_vae:
        _z = 0.5 * torch.randn(1, 4, latent, latent, device=device)
        z_stage1 = 0.5 * torch.randn(1, 4, latent, latent, device=device)
    else:
        _z = m.encode_first_stage_with_denoise(img, use_sample=False)
        x_stage1 = m.decode_first_stage(_z)
        z_stage1 = m.encode_first_stage(x_stage1)
        del x_stage1
    e2.record()
    barrier()
    h2d_img_ms, vae_pre_ms = e0.elapsed_time(e1), e1.elapsed_time(e2)
    del img
    cond, ucond = dict(c, control=_z), dict(uc, control=_z)
    noised = torch.randn_like(_z)
    smp = m.make_sampler(w["steps"], -1.0, 5, 1.01, 4.0, True, 1.0)
    denoiser = sampling.FusedDenoiser(m.denoiser, net)
    run = smp.begin(denoiser, noised, cond, ucond, x_center=z_stage1, control_scale=1.0)
    nsteps = run.num_steps

    # ---- warm-up steps (graph capture happens in the first one) ----
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    for i in range(args.warmup):
        run.step(i % nsteps)
    barrier()
    # ---- timed region: EXACTLY K sampler steps (device-resident) ----
    clocks.mark()
    lc0 = _native.launch_count() + net.replayed_launches
    barrier()
    prof = os.environ.get("SUPIR_BENCH_CUDA_PROFILER", "0") == "1"     # `ncu --profile-from-start off`: capture the timed steps only
    t0, t1 = ev(), ev()
    if prof:
        torch.cuda.profiler.start()
    t0.record()
    for i in range(args.warmup, args.warmup + args.steps):
        run.step(i % nsteps)
    t1.record()
    barrier()
    if prof:
        torch.cuda.profiler.stop()
    step_ms = t0.elapsed_time(t1) / args.steps
    lc1 = _native.launch_count() + net.replayed_launches
    clk = clocks.stop() if rank == 0 else None
    # the latent the last timed sampler step returned; the e2e steps below overwrite run.x
    dumped = run.x.detach().float().cpu() if args.dump_outputs else None
    # ---- e2e steps: host latent in, host latent out, every step ----
    x_host = run.x.detach().cpu().pin_memory()
    res_host = torch.empty_like(x_host).pin_memory()
    barrier()
    t2, t3 = ev(), ev()
    t2.record()
    for i in range(args.warmup + args.steps, args.warmup + 2 * args.steps):
        run.x.copy_(x_host, non_blocking=True)
        run.step(i % nsteps)
        res_host.copy_(run.x, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    t3.record()
    barrier()
    e2e_step_ms = t2.elapsed_time(t3) / args.steps
    # ---- final decode (SUPIR_model.py:131) + image download ----
    e3, e4, e5 = ev(), ev(), ev()
    e3.record()
    samples = m.decode_first_stage(run.x) if not skip_vae else torch.zeros(1, 3, 8, 8, device=device)
    e4.record()
    if not skip_vae:
        out_host.copy_(samples, non_blocking=True)
    e5.record()
    barrier()
    vae_post_ms, d2h_img_ms = e3.elapsed_time(e4), e4.elapsed_time(e5)
    finite = bool(torch.isfinite(samples).all())
    del samples, run

    # ---- ONE real run of the whole configuration through SUPIRModel.batchify_sample, host image in -> host image out ----
    full = None
    if not skip_vae and not args.no_full_run:
        barrier()
        tw0 = time.perf_counter()
        f0, f1 = ev(), ev()
        f0.record()
        res = m.batchify_sample(img_host.to(device, non_blocking=True), num_steps=w["steps"], restoration_scale=-1.0, s_churn=5, s_noise=1.01,
                                cfg_scale=4.0, seed=1234 if w["shards"] else 1234 + rank, control_scale=1.0, use_linear_CFG=True,
                                cfg_scale_start=1.0, c=c, uc=uc)
        out_host.copy_(res, non_blocking=True)
        f1.record()
        barrier()
        full = {"device_s": f0.elapsed_time(f1) / 1e3, "wall_s": time.perf_counter() - tw0, "finite": bool(torch.isfinite(res).all())}
        del res

    def maxr(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    step_ms, e2e_step_ms = maxr(step_ms), maxr(e2e_step_ms)
    vae_pre_ms, vae_post_ms = maxr(vae_pre_ms), maxr(vae_post_ms)
    vae_ms = vae_pre_ms + vae_post_ms
    xfer_ms = maxr(h2d_img_ms) + maxr(d2h_img_ms)
    if full is not None:
        full["device_s"], full["wall_s"] = maxr(full["device_s"]), maxr(full["wall_s"])
        full["mp_per_s"] = megapixels / full["wall_s"]
        full["what"] = "one SUPIRModel.batchify_sample call (2 encodes, %d sampler steps, 2 decodes), pinned host image in, host image out, max over ranks" % w["steps"]
    total_s = (w["steps"] * step_ms + vae_ms) / 1e3
    e2e_total_s = (w["steps"] * e2e_step_ms + vae_ms + xfer_ms) / 1e3
    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    # ---- roofline of the dominant kernel + CPU baseline (rank 0, N = 1 only) ----
    roof, cpu = None, None
    prof = profile_dominant_kernel(net, device)
    traffic, traffic_src = load_traffic()
    ranks_on_step = world if shards else 1
    if prof is not None:
        g_flops, g_ms, g_n, g_key = prof
        achieved = g_flops / (g_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "kernel": "supir::gemm_tcgen05_kernel (Linear / conv1x1 / implicit-GEMM conv3x3)",
                "achieved": achieved, "peak": sust, "peak_kind": f"bf16 dense sustained, {peak_kind}", "unit": "TFLOP/s",
                "frac": achieved / sust, "traffic": traffic, "traffic_unit": f"bytes/launch (mean of the ncu --set full capture profiles/{traffic_src})",
                "launches_timed": g_n, "plan_batch_h_w_ctx": list(g_key),
                "step_flops": step_flop, "step_achieved_tflops": step_flop / (step_ms * 1e-3) / 1e12,
                "step_frac_of_peak": step_flop / (step_ms * 1e-3) / 1e12 / (sust * ranks_on_step)}
    if world == 1 and not args.no_cpu_baseline:
        cores = min(os.cpu_count() or 1, int(os.environ.get("SUPIR_BENCH_CPU_THREADS", "64")))
        torch.set_num_threads(cores)
        sd = oracle_state_dict(fast=True)
        budget = float(os.environ.get("SUPIR_BENCH_CPU_BUDGET_S", "30"))
        sec_window, meas, how = probe_oracle_window(sd, budget * 0.8, 1)
        del sd
        enc_s, dec_s, vae_note = time_oracle_vae(budget * 0.2, 1088, 150)
        cpu_total_s, _, _ = cpu_model(args.config, sec_window, enc_s, dec_s)
        cpu = {"value": megapixels / cpu_total_s, "unit": "MP/s", "cores": cores, "kind": "port",
               "sample": f"oracle (fp32, {cores} threads) control+UNet on one 128x128-latent window (CFG pair): {how} {sec_window:.2f} s "
                         f"(probes 32: {meas[32][0]:.2f} s, 64: {meas[64][0]:.2f} s); VAE: {vae_note}; job extrapolated: {windows} window(s) x "
                         f"{w['steps']} steps + 2 encodes + 2 decodes = {cpu_total_s:.0f} s"}
    line = {
        "metric": "megapixels_per_sec", "value": megapixels / total_s, "unit": "MP/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "strong" if w["shards"] else "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"{args.config}: " + w["desc"] + "; SUPIR-v0 + SDXL-base + SDXL-VAE shapes, random weights",
                   "sampler_steps": w["steps"], "windows": windows, "tile_batch": getattr(smp, "tile_batch", None), "images": images,
                   "vae_ms": vae_ms, "vae_pre_ms": vae_pre_ms, "vae_post_ms": vae_post_ms, "vae_warmup_passes": min(args.warmup, 1), "vae_warmup": "one untimed denoise-encode + decode + encode (fills the three networks' scratch pools)",
                   "l2": "per-step working set (7.7 GB of weights + activations) exceeds the 126 MB L2",
                   "output_finite": finite, "vae_skipped_INVALID_FOR_BENCH": skip_vae,
                   "parallelism": (f"(CFG branch, window) units and VAE tiles sharded over {world} rank(s), 1 all-gather/step" if shards else
                                   (f"{world} independent replicas" if world > 1 else "single GPU"))},
        "ms_per_edm_step": step_ms,
        "e2e": {"value": megapixels / e2e_total_s, "unit": "MP/s", "ms_per_step": e2e_step_ms,
                "h2d_bytes_per_step": int(x_host.numel() * 4), "d2h_bytes_per_step": int(res_host.numel() * 4),
                "image_h2d_bytes": int(img_host.numel() * 4), "image_d2h_bytes": int(out_host.numel() * 4)},
        "full_run": full,
        "gpu_launches": int(lc1 - lc0),
        "clocks": clk,
        "roofline": roof,
    }
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "latent.npy"), dumped.numpy())
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="supir_b200", choices=["supir_b200", "reference"])
    ap.add_argument("--config", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-full-run", action="store_true", help="skip the one real batchify_sample run of the whole configuration")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the latent the last timed sampler step returned to DIR/latent.npy (float32; rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "supir_b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the supir_b200 arm has no CPU fallback (use --impl reference for the CPU oracle)")
        run_supir(args)


if __name__ == "__main__":
    main()

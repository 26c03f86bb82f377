"""The drop-in claim, end to end, on CPU: this package's engine (supir_b200.model.SUPIRModel) is built from a YAML-shaped config
and the same weights as the reference's own engine class (SUPIR/models/SUPIR_model.py `SUPIRModel(DiffusionEngine)`), and
`batchify_sample(image, prompts, ...)` is run: stage-1 encode / decode, re-encode, text conditioning from prompt strings, the EDM
restore sampler, final decode, also with the tiled VAE hooks (`init_tile_vae`), the tiled sampler and per-window prompts, then the
stage-1-only denoise. The reference engine's outputs on the same config, weights, inputs and noise sequence (a fixed seeded sample
of each, with its shape) are stored in
tests/golden/dropin_engine.npz (tests/golden/make_reference_io.py), together with its state_dict layout and sigma table.
No GPU here, so the backend's kernels are the plain-torch stand-ins of tests/cpu_ops.py (bf16 storage where the kernels store
bf16): what this pins is the engine's state_dict layout, its call signatures and RNG order, and that it produces the reference's
result within the bf16 tolerance."""
import copy
import json
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import reference_cases  # noqa: E402
from weights import cond_tokens, make_state_dict, randn  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "dropin_engine.npz")
WEIGHT_SEED = 123
DISC = {"target": "sgm.modules.diffusionmodules.discretizer.LegacyDDPMDiscretization"}
# full SDXL widths (LightGLVUNet's 'XL-base' adapter tables are hard-coded for 320 / 640 / 1280 channels, SUPIR_v0.py:560-598) with
# depth-1 transformers, and both text towers at their real widths with two blocks each: 980 M + 145 M parameters per engine
NET = dict(adm_in_channels=2816, num_classes="sequential", use_checkpoint=True, in_channels=4, out_channels=4, model_channels=320,
           attention_resolutions=[4, 2], num_res_blocks=2, channel_mult=[1, 2, 4], num_head_channels=64, use_spatial_transformer=True,
           use_linear_in_transformer=True, transformer_depth=[1, 1, 1], context_dim=2048, spatial_transformer_attn_type="softmax-xformers",
           legacy=False)
VAE = dict(attn_type="vanilla", double_z=True, z_channels=4, resolution=64, in_channels=3, out_ch=3, ch=32, ch_mult=[1, 2, 4, 4],
           num_res_blocks=1, attn_resolutions=[], dropout=0.0)
ARCH_L = dict(vocab=49408, width=768, heads=12, layers=2, mlp=3072, ctx=77, act="quick_gelu", eps=1e-5)
ARCH_G = dict(vocab=49408, width=1280, heads=20, layers=2, mlp=5120, ctx=77, proj=1280, act="gelu", eps=1e-5)
EMB = [
    {"is_trainable": False, "input_key": "txt", "target": "sgm.modules.encoders.modules.FrozenCLIPEmbedder",
     "params": {"layer": "hidden", "layer_idx": 1, "arch": {"layers": 2}}},
    {"is_trainable": False, "input_key": "txt", "target": "sgm.modules.encoders.modules.FrozenOpenCLIPEmbedder2",
     "params": {"arch": "ViT-bigG-14", "layer": "penultimate", "always_return_pooled": True, "legacy": False, "text_cfg": {"layers": 2}}}]
EMB += [{"is_trainable": False, "input_key": k, "target": "sgm.modules.encoders.modules.ConcatTimestepEmbedderND", "params": {"outdim": 256}}
        for k in ("original_size_as_tuple", "crop_coords_top_left", "target_size_as_tuple")]


class Cfg(dict):
    """OmegaConf stand-in (the package is absent): nested dicts with attribute access, which batchify_sample uses
    (`self.sampler_config.params.num_steps = ...`, SUPIR_model.py:101-111)."""

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:
            raise AttributeError(k) from e

    def __setattr__(self, k, v):
        self[k] = v

    def __deepcopy__(self, memo):
        return cfgify({k: copy.deepcopy(v, memo) for k, v in self.items()})


def cfgify(d):
    if isinstance(d, dict):
        return Cfg({k: cfgify(v) for k, v in d.items()})
    if isinstance(d, (list, tuple)):
        return [cfgify(v) for v in d]
    return d


def engine_config(sampler_target, with_conditioner, extra=None):
    return cfgify(dict(
        control_stage_config={"target": "SUPIR.modules.SUPIR_v0.GLVControl", "params": dict(NET, input_upscale=1)},
        network_config={"target": "SUPIR.modules.SUPIR_v0.LightGLVUNet", "params": dict(NET, mode="XL-base", project_type="ZeroSFT", project_channel_scale=2)},
        network_wrapper="sgm.modules.diffusionmodules.wrappers.ControlWrapper",
        denoiser_config={"target": "sgm.modules.diffusionmodules.denoiser.DiscreteDenoiserWithControl",
                         "params": {"num_idx": 1000, "weighting_config": {"target": "sgm.modules.diffusionmodules.denoiser_weighting.EpsWeighting"},
                                    "scaling_config": {"target": "sgm.modules.diffusionmodules.denoiser_scaling.EpsScaling"},
                                    "discretization_config": DISC}},
        first_stage_config={"target": "sgm.models.autoencoder.AutoencoderKLInferenceWrapper",
                            "params": {"embed_dim": 4, "ddconfig": VAE, "lossconfig": {"target": "torch.nn.Identity"}}},
        conditioner_config=({"target": "sgm.modules.GeneralConditionerWithControl", "params": {"emb_models": EMB}} if with_conditioner else None),
        sampler_config={"target": sampler_target,
                        "params": dict({"num_steps": 100, "restore_cfg": 4.0, "s_churn": 0, "s_noise": 1.003, "device": "cpu", "discretization_config": DISC,
                                        "guider_config": {"target": "sgm.modules.diffusionmodules.guiders.LinearCFG", "params": {"scale": 7.5, "scale_min": 4.0}}},
                                       **(extra or {}))},
        ae_dtype="bf16", diffusion_dtype="bf16", scale_factor=0.13025, p_p=", best quality", n_p="blurry"))


def prompt_row(text, pad):
    import zlib
    return cond_tokens(zlib.crc32(text.encode()) % 100000, 1, 49408, pad)[0]


class SeededNoise:
    def __init__(self, base):
        self.base, self.n = base, 0

    def __call__(self, x, **k):
        self.n += 1
        return randn(tuple(x.shape), self.base + self.n).to(x.dtype)


def rel_fro(a, b):
    return float((a - b).norm() / b.norm())


@pytest.fixture()
def backend_on_standins(monkeypatch):
    """CPU stand-in kernels + the three `needs CUDA` guards lifted; monkeypatch puts everything back."""
    sys.path.insert(0, HERE)
    import cpu_ops
    from supir_b200 import ops, vae, wrappers
    cpu_ops.install(monkeypatch)
    monkeypatch.setattr(vae._VAENet, "_check", lambda self, x: (None if getattr(self, "_packed", False) else self.pack()))

    def conv1x1(self, x, in_scale=1.0):
        x = x.float().contiguous()
        out = torch.empty((x.shape[0], self.out_channels) + tuple(x.shape[2:]), dtype=torch.float32)
        w = self.weight.detach().reshape(self.out_channels, self.in_channels).to(torch.bfloat16).float().contiguous()
        return ops.conv1x1_small_nchw(x, w, vae._bias_bf16_values(self.bias), out, in_scale=in_scale)
    monkeypatch.setattr(vae._Conv1x1Small, "forward", conv1x1)

    def wrapper_forward(self, x, t, c, control_scale=1, context_token=None, **kw):      # ControlWrapper.forward minus the CUDA graph
        if not self._packed:
            self.pack()
        ctx, y = c["crossattn"], c["vector"]
        plan = wrappers._Plan(self, x.shape[0], x.shape[2], x.shape[3], ctx.shape[1], ctx.shape[2], y.shape[1], "cpu")
        wrappers.ControlWrapper._fill(plan, x, t, ctx, y, c["control"], control_scale, context_token)
        plan._run()
        return plan.out.clone()
    monkeypatch.setattr(wrappers.ControlWrapper, "forward", wrapper_forward)


SAMPLING = "sgm.modules.diffusionmodules.sampling."
P_P, N_P = ", best quality", "blurry"
LOCAL = ["a cat", "a dog on grass", "sky", "a red brick wall"]          # 24 x 24 latent, tile 16 / stride 8 -> 4 windows
# (name, sampler target, extra sampler params, tiled VAE, image size, prompts): `tiled_local_prompts` passes one prompt per
# sampler window, the way gradio_demo_tiled.py does (p = [[...]], SUPIR_model.py:163-176 -> a list of conds, sampling.py:623-627)
SCENARIOS = [("untiled", "RestoreEDMSampler", None, False, 128, ["a photo of a cat"]),
             ("tiled_local_prompts", "TiledRestoreEDMSampler", {"tile_size": 16, "tile_stride": 8}, True, 192, [LOCAL])]
KW = dict(num_steps=2, restoration_scale=4.0, s_churn=5, s_noise=1.01, cfg_scale=4.0, seed=77, control_scale=0.9,
          use_linear_CFG=True, cfg_scale_start=1.0, use_linear_control_scale=True, control_scale_start=0.3)


def run_scenarios(eng, monkeypatch, untile_reference_hooks=False):
    """batchify_sample for every scenario on ONE engine (the sampler is rebuilt per call from `sampler_config`, which test.py /
    the demos also overwrite between calls), then the stage-1-only path of gradio_demo*.py through a second denoise encoder."""
    out = {}
    for name, target, extra, tiled_vae, size, prompts in SCENARIOS:
        eng.sampler_config = engine_config(SAMPLING + target, False, extra)["sampler_config"]
        if tiled_vae and not getattr(eng, "_tile_vae_on", False):
            eng.init_tile_vae(encoder_tile_size=64, decoder_tile_size=8)
            eng._tile_vae_on = True
            if untile_reference_hooks:
                for net in (eng.first_stage_model.denoise_encoder, eng.first_stage_model.encoder, eng.first_stage_model.decoder):
                    net.forward.to_gpu = False                  # VAEHook(to_gpu=True) moves the net to devices.get_optimal_device()
        img = (randn((1, 3, size, size), 500) * 0.5).clamp(-1, 1)
        monkeypatch.setattr(torch, "randn_like", SeededNoise(9000))
        out[name] = eng.batchify_sample(img, list(prompts), **KW)
    eng.first_stage_model.denoise_encoder_s1 = copy.deepcopy(eng.first_stage_model.denoise_encoder)
    out["stage1_denoise"] = eng.batchify_denoise(img, is_stage1=True)       # gradio_demo_tiled.py:54, 95 (tiled hooks in place)
    return out


def prompt_tokens():
    """Token ids of every prompt the scenarios use (both towers), in place of the BPE tokenisers."""
    texts = ["a photo of a cat" + P_P] + [t + P_P for t in LOCAL] + [N_P]
    return {t: prompt_row(t, 49407) for t in texts}, {t: prompt_row(t, 0) for t in texts}


def test_engine_matches_the_reference_engine(backend_on_standins, monkeypatch):
    import contextlib
    import io
    import warnings
    from supir_b200.model import SUPIRModel
    ref = np.load(GOLDEN)
    shapes = json.loads(str(ref["shapes"]))
    tok_l, tok_g = prompt_tokens()
    with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        eng = SUPIRModel(**engine_config(SAMPLING + "RestoreEDMSampler", True)).eval()
        assert type(eng.model).__module__ == "supir_b200.wrappers" and type(eng.conditioner).__module__ == "supir_b200.conditioner"
        assert type(eng.first_stage_model).__module__ == "supir_b200.vae" and type(eng.denoiser).__module__ == "supir_b200.denoiser"
        assert {k: list(v.shape) for k, v in eng.state_dict().items()} == shapes, "state_dict layout differs from the reference engine's"
        sd = make_state_dict(shapes, seed=WEIGHT_SEED)
        sd["denoiser.sigmas"] = torch.from_numpy(ref["sigmas"])  # a persistent buffer, not a weight: keep the real sigma table
        eng.load_state_dict(sd)
        eng.conditioner.embedders[0].tokenize = lambda ts: torch.stack([tok_l[t] for t in ts])
        eng.conditioner.embedders[1].tokenize = lambda ts: torch.stack([tok_g[t] for t in ts])
        got = run_scenarios(eng, monkeypatch)
        assert type(eng.sampler).__module__ == "supir_b200.sampling" and type(eng.first_stage_model.decoder.forward).__module__ == "supir_b200.vae"
    assert sorted(got) == sorted(k for k in ref.files if k + "_shape" in ref.files)
    errs = {k: rel_fro(reference_cases.sample(got[k]), torch.from_numpy(ref[k])) for k in got}
    print("SUPIRModel on the backend, rel. Frobenius vs the reference engine (seeded sample):", {k: f"{v:.4g}" for k, v in errs.items()})
    for k, v in errs.items():
        assert list(got[k].shape) == ref[k + "_shape"].tolist() and v <= (3e-2 if k == "stage1_denoise" else 5e-2), (k, v)

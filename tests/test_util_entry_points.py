"""supir_b200.util's model-construction entry points (SUPIR/util.py:11-57: create_SUPIR_model / load_QF_ckpt / load_state_dict /
convert_dtype — what test.py and the gradio demos import) on synthetic checkpoints in both on-disk formats, driven by a YAML
file with the layout of options/SUPIR_v0.yaml; and the small numpy helpers against the reference's own functions."""
import os
import sys

import numpy as np
import pytest
import torch
import yaml

from weights import make_state_dict

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))

DISC = {"target": "sgm.modules.diffusionmodules.discretizer.LegacyDDPMDiscretization"}
# construction + checkpoint loading only (no forward pass): a narrow network keeps the files small
NET = dict(adm_in_channels=64, num_classes="sequential", use_checkpoint=False, in_channels=4, out_channels=4, model_channels=64,
           attention_resolutions=[4, 2], num_res_blocks=2, channel_mult=[1, 2, 4], num_head_channels=64, use_spatial_transformer=True,
           use_linear_in_transformer=True, transformer_depth=[1, 1, 2], context_dim=48, spatial_transformer_attn_type="softmax-xformers", legacy=False)
VAE = dict(attn_type="vanilla-xformers", double_z=True, z_channels=4, resolution=64, in_channels=3, out_ch=3, ch=32, ch_mult=[1, 2],
           num_res_blocks=1, attn_resolutions=[], dropout=0.0)


def write_config(tmp_path):
    model = {"target": "SUPIR.models.SUPIR_model.SUPIRModel", "params": dict(
        ae_dtype="bf16", diffusion_dtype="bf16", scale_factor=0.13025, network_wrapper="sgm.modules.diffusionmodules.wrappers.ControlWrapper",
        control_stage_config={"target": "SUPIR.modules.SUPIR_v0.GLVControl", "params": dict(NET, input_upscale=1)},
        network_config={"target": "SUPIR.modules.SUPIR_v0.LightGLVUNet", "params": dict(NET, mode="XL-base", project_type="ZeroSFT", project_channel_scale=2)},
        denoiser_config={"target": "sgm.modules.diffusionmodules.denoiser.DiscreteDenoiserWithControl",
                         "params": {"num_idx": 1000, "weighting_config": {"target": "sgm.modules.diffusionmodules.denoiser_weighting.EpsWeighting"},
                                    "scaling_config": {"target": "sgm.modules.diffusionmodules.denoiser_scaling.EpsScaling"}, "discretization_config": DISC}},
        first_stage_config={"target": "sgm.models.autoencoder.AutoencoderKLInferenceWrapper",
                            "params": {"ckpt_path": None, "embed_dim": 4, "monitor": "val/rec_loss", "ddconfig": VAE, "lossconfig": {"target": "torch.nn.Identity"}}},
        sampler_config={"target": "sgm.modules.diffusionmodules.sampling.RestoreEDMSampler",
                        "params": {"num_steps": 100, "restore_cfg": 4.0, "s_churn": 0, "s_noise": 1.003, "discretization_config": DISC,
                                   "guider_config": {"target": "sgm.modules.diffusionmodules.guiders.LinearCFG", "params": {"scale": 7.5, "scale_min": 4.0}}}},
        p_p="Cinematic, High Contrast", n_p="painting, oil painting")}
    cfg = {"model": model, "SDXL_CKPT": str(tmp_path / "sdxl.safetensors"), "SUPIR_CKPT_F": str(tmp_path / "v0F.ckpt"),
           "SUPIR_CKPT_Q": str(tmp_path / "v0Q.ckpt"), "SUPIR_CKPT": None,
           "default_setting": {"s_cfg_Quality": 7.5, "spt_linear_CFG_Quality": 4.0, "s_cfg_Fidelity": 4.0, "spt_linear_CFG_Fidelity": 1.0, "edm_steps": 50}}
    path = tmp_path / "SUPIR_v0.yaml"
    with open(path, "w") as f:
        yaml.safe_dump(cfg, f)
    return str(path), cfg


def test_create_supir_model_loads_both_checkpoint_formats_in_the_reference_order(tmp_path):
    import safetensors.torch
    from supir_b200 import util
    from supir_b200.config import instantiate_from_config
    path, cfg = write_config(tmp_path)
    probe = instantiate_from_config(cfg["model"])
    shapes = {k: list(v.shape) for k, v in probe.state_dict().items()}
    base = make_state_dict(shapes, seed=1)
    base["denoiser.sigmas"] = probe.denoiser.sigmas.clone()
    # SDXL file: everything but the control net and the adapters; SUPIR Q / F files: control net + adapters, wrapped in 'state_dict'
    is_supir = lambda k: k.startswith("model.control_model.") or ".project_modules." in k  # noqa: E731
    safetensors.torch.save_file({k: v.contiguous() for k, v in base.items() if not is_supir(k)}, cfg["SDXL_CKPT"])
    q = {k: v for k, v in make_state_dict(shapes, seed=2).items() if is_supir(k)}
    f_ = {k: v for k, v in make_state_dict(shapes, seed=3).items() if is_supir(k)}
    torch.save({"state_dict": q}, cfg["SUPIR_CKPT_Q"])
    torch.save(f_, cfg["SUPIR_CKPT_F"])                               # both wrappings occur in the wild
    assert q and len(q) < len(base)
    model, default_setting = util.create_SUPIR_model(path, SUPIR_sign="Q", load_default_setting=True)
    assert type(model).__module__ == "supir_b200.model" and default_setting.s_cfg_Quality == 7.5 and default_setting.edm_steps == 50
    got = model.state_dict()
    for k in shapes:
        want = q[k] if is_supir(k) else base[k]
        assert torch.equal(got[k], want), k
    assert model.p_p == "Cinematic, High Contrast" and model.model.dtype == torch.bfloat16 and model.ae_dtype == torch.bfloat16
    model_f = util.create_SUPIR_model(path, SUPIR_sign="F")
    assert all(torch.equal(model_f.state_dict()[k], f_[k]) for k in f_)
    ckpt_q, ckpt_f = util.load_QF_ckpt(path)
    assert set(get_keys(ckpt_q)) == set(q) and set(get_keys(ckpt_f)) == set(f_)
    model.load_state_dict(util.get_state_dict(ckpt_f), strict=False)   # the run-time switch of gradio_demo*.py
    assert all(torch.equal(model.state_dict()[k], f_[k]) for k in f_)
    assert util.convert_dtype("fp16") is torch.float16 and util.convert_dtype("bf16") is torch.bfloat16
    with pytest.raises(NotImplementedError):
        util.convert_dtype("int8")


def get_keys(ckpt):
    return ckpt.get("state_dict", ckpt).keys()


def test_numpy_helpers_match_the_reference_functions():
    """HWC3 / Numpy2Tensor against the reference's own functions (SUPIR/util.py), through their recorded outputs
    (tests/golden/reference_io.npz)."""
    import reference_cases
    from supir_b200 import util
    ref = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_io.npz"))
    imgs, img = reference_cases.numpy_helper_inputs()
    for i, x in enumerate(imgs):
        want = ref[f"hwc3_{i}"]
        got = util.HWC3(x)
        assert got.dtype == want.dtype and np.array_equal(got, want)
    got = util.Numpy2Tensor(img)
    assert got.numpy().dtype == ref["numpy2tensor"].dtype and np.array_equal(got.numpy(), ref["numpy2tensor"])

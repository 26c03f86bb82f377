"""compat.install() against the reference's module layout, the reference's model configurations through this package's factory,
and PreparedConditioner against the reference class. The reference is not part of this repository: its three configurations are
stored unedited under tests/golden/options/, and the names its modules define and what its PreparedConditioner returns are
recorded in tests/golden/reference_io.npz (tests/golden/make_reference_io.py)."""
import importlib
import json
import os
import sys
import types

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
sys.path.insert(0, GOLDEN)
REF =np.load(os.path.join(GOLDEN, "reference_io.npz"))
REF_NAMES = json.loads(str(REF["compat_names"]))


@pytest.fixture()
def reference_modules(monkeypatch):
    """Stand-ins for the reference modules compat.install() patches, each holding a placeholder under every name the reference's
    module defines; they leave sys.modules when the test ends."""
    placeholders = {}
    for modname, attrs in REF_NAMES.items():
        parts = modname.split(".")
        for i in range(1, len(parts) + 1):
            name = ".".join(parts[:i])
            if name not in placeholders:
                monkeypatch.setitem(sys.modules, name, types.ModuleType(name))
                placeholders[name] = {}
        mod = sys.modules[modname]
        for a in attrs:
            placeholders[modname][a] = type(a, (), {"__module__": modname})
            setattr(mod, a, placeholders[modname][a])
    return placeholders


def test_install_rebinds_reference_targets(reference_modules):
    import supir_b200.compat as compat
    for modname, attrs in dict(compat.PATCHES, **compat.CONDITIONER_PATCHES).items():
        assert set(attrs) <= set(REF_NAMES[modname]), f"compat patches names {modname} does not define"
    done = compat.install(strict=False)
    assert sorted(done) == sorted((m, a) for m, attrs in compat.PATCHES.items() for a in attrs)
    for m, a in done:
        assert getattr(importlib.import_module(m), a) is compat._resolve(compat.PATCHES[m][a])
    # what the reference's get_obj_from_str / instantiate_from_config do with a target string: import the module, getattr
    smp_cls = getattr(importlib.import_module("sgm.modules.diffusionmodules.sampling"), "TiledRestoreEDMSampler")
    smp = smp_cls(num_steps=5, restore_cfg=4.0, s_churn=0, s_noise=1.003, tile_size=128, tile_stride=64, device="cpu",
                  discretization_config={"target": "sgm.modules.diffusionmodules.discretizer.LegacyDDPMDiscretization"},
                  guider_config={"target": "sgm.modules.diffusionmodules.guiders.LinearCFG", "params": {"scale": 7.5, "scale_min": 4.0}})
    assert type(smp).__module__ == "supir_b200.sampling" and type(smp.guider).__module__ == "supir_b200.guiders"
    assert getattr(importlib.import_module("SUPIR.modules.SUPIR_v0"), "GLVControl").__module__ == "supir_b200.nets"
    assert getattr(importlib.import_module("sgm.modules.diffusionmodules.wrappers"), "ControlWrapper").__module__ == "supir_b200.wrappers"


def test_install_conditioner_is_opt_in_and_resolves_through_the_reference_factory(reference_modules):
    import supir_b200.compat as compat
    E = importlib.import_module("sgm.modules.encoders.modules")
    compat.install(strict=False)
    assert E.FrozenCLIPEmbedder is reference_modules["sgm.modules.encoders.modules"]["FrozenCLIPEmbedder"]   # untouched by default
    compat.install(strict=False, conditioner=True)
    assert getattr(importlib.import_module("sgm.modules"), "GeneralConditionerWithControl").__module__ == "supir_b200.conditioner"
    assert getattr(E, "FrozenOpenCLIPEmbedder2").__module__ == "supir_b200.conditioner"


def test_every_reference_yaml_instantiates_through_this_packages_factory():
    """options/SUPIR_v0.yaml, SUPIR_v0_tiled.yaml and SUPIR_v0_Juggernautv9_lightning.yaml, unedited: every `target:` string of the
    model section — engine, wrapper, denoiser, both networks, VAE, sampler + guider, the conditioner with both text towers at
    full size — resolves to this package's classes (built on the meta device: 4.8 B parameters cost nothing)."""
    import glob
    import torch
    from supir_b200.config import instantiate_from_config, load_yaml
    paths = sorted(glob.glob(os.path.join(GOLDEN, "options", "*.yaml")))
    assert len(paths) >= 3
    samplers = set()
    for path in paths:
        cfg = load_yaml(path, attr_access=True)
        with torch.device("meta"):
            m = instantiate_from_config(cfg.model)
        mods = {type(x).__module__ for x in (m, m.model, m.model.diffusion_model, m.model.control_model, m.denoiser, m.sampler, m.sampler.guider,
                                             m.first_stage_model, m.conditioner, *m.conditioner.embedders)}
        assert all(x.startswith("supir_b200.") for x in mods), (path, mods)
        keys = m.state_dict().keys()
        assert sum(k.startswith("conditioner.embedders.0.transformer.text_model.encoder.layers.") for k in keys) == 12 * 16
        assert sum(k.startswith("conditioner.embedders.1.model.transformer.resblocks.") for k in keys) == 32 * 12
        assert sum(p.numel() for p in m.model.parameters()) > 3.8e9
        assert cfg.SDXL_CKPT and cfg.SUPIR_CKPT_Q
        samplers.add(type(m.sampler).__name__)
    assert samplers == {"RestoreEDMSampler", "TiledRestoreEDMSampler", "RestoreDPMPP2MSampler"}


def test_prepared_conditioner_matches_the_reference_class(tmp_path):
    """sgm.modules.PreparedConditioner (modules.py:246-290): conditions loaded from .pth files and repeated to the batch."""
    import torch
    import reference_cases
    from supir_b200.config import instantiate_from_config
    c, uc, batch = reference_cases.prepared_conditioner_inputs()
    torch.save(c, tmp_path / "c.pth")
    torch.save(uc, tmp_path / "uc.pth")
    for tag, un in (("uc", str(tmp_path / "uc.pth")), ("none", None)):
        mine = instantiate_from_config({"target": "sgm.modules.PreparedConditioner", "params": {"cond_pth": str(tmp_path / "c.pth"), "un_cond_pth": un}})
        assert type(mine).__module__ == "supir_b200.conditioner"
        a, au = mine.get_unconditional_conditioning(batch)
        want = {k[len(f"prepared_{tag}_c_"):]: REF[k] for k in REF.files if k.startswith(f"prepared_{tag}_c_")}
        want_u = {k[len(f"prepared_{tag}_uc_"):]: REF[k] for k in REF.files if k.startswith(f"prepared_{tag}_uc_")}
        assert sorted(a) == sorted(want) and all(np.array_equal(a[k].numpy(), want[k]) for k in a)
        assert (au is None and not want_u) or (sorted(au) == sorted(want_u) and all(np.array_equal(au[k].numpy(), want_u[k]) for k in au))
        assert sorted(mine.state_dict().keys()) == json.loads(str(REF[f"prepared_{tag}_keys"]))

"""Record what the reference returns for the inputs of the tests that compare this package with it directly.

The reference is not part of this repository, so those tests compare with these stored outputs instead of calling it:
  reference_io.npz        PIL2Tensor digests, HWC3 / Numpy2Tensor outputs, PreparedConditioner outputs, the names compat.install
                          rebinds, and digests of the integer bookkeeping on seeded random sizes (tests/test_properties.py)
  dropin_engine.npz       SUPIRModel.batchify_sample / batchify_denoise of the reference engine (tests/test_dropin_reference_engine_cpu.py)
  options/*.yaml          the reference's three model configurations, unedited

Run with a checkout of the reference at $SUPIR_REFERENCE_ROOT:   python tests/golden/make_reference_io.py [io] [engine] [options]
"""
import contextlib
import io
import json
import os
import shutil
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
for p in (HERE, TESTS, os.path.dirname(TESTS)):
    if p not in sys.path:
        sys.path.insert(0, p)

import ref_stubs  # noqa: E402
import reference_cases as cases  # noqa: E402


def _exec_ref_functions(first, stop, ns):
    with open(os.path.join(ref_stubs.REFERENCE_ROOT, "SUPIR", "util.py")) as f:
        src = f.read()
    exec(src[src.index(first):src.index(stop)], ns)
    return ns


def gen_io():
    from PIL import Image
    ref = ref_stubs.import_reference()
    out = {}

    # PIL2Tensor (SUPIR/util.py): the tensor's digest and the reported size, per image and argument set
    ns = _exec_ref_functions("def PIL2Tensor", "def Tensor2PIL", {"np": np, "torch": torch, "Image": Image})
    rows = []
    for img, args in cases.pil2tensor_cases(Image):
        t, h0, w0 = ns["PIL2Tensor"](img, **args)
        rows.append([cases.digest(t), h0, w0])
    out["pil2tensor"] = np.array(json.dumps(rows))

    # HWC3 / Numpy2Tensor
    ns = _exec_ref_functions("def HWC3", "def upscale_image", {"np": np, "torch": torch})
    _exec_ref_functions("def Numpy2Tensor", "def Tensor2Numpy", ns)
    imgs, img = cases.numpy_helper_inputs()
    for i, x in enumerate(imgs):
        out[f"hwc3_{i}"] = ns["HWC3"](x)
    out["numpy2tensor"] = ns["Numpy2Tensor"](img).numpy()

    # PreparedConditioner: conditions from .pth files, repeated to the batch
    import importlib
    import tempfile
    E = importlib.import_module("sgm.modules.encoders.modules")
    c, uc, batch = cases.prepared_conditioner_inputs()
    with tempfile.TemporaryDirectory() as d:
        torch.save(c, os.path.join(d, "c.pth"))
        torch.save(uc, os.path.join(d, "uc.pth"))
        for tag, un in (("uc", os.path.join(d, "uc.pth")), ("none", None)):
            m = E.PreparedConditioner(os.path.join(d, "c.pth"), un)
            a, au = m.get_unconditional_conditioning(batch)
            out.update({f"prepared_{tag}_c_{k}": v.numpy() for k, v in a.items()})
            if au is not None:
                out.update({f"prepared_{tag}_uc_{k}": v.numpy() for k, v in au.items()})
            out[f"prepared_{tag}_keys"] = np.array(json.dumps(sorted(m.state_dict().keys())))

    # the attributes compat.install rebinds, as the reference's modules define them
    import supir_b200.compat as compat
    names = {}
    for modname, attrs in dict(compat.PATCHES, **compat.CONDITIONER_PATCHES).items():
        mod = importlib.import_module(modname)
        names[modname] = sorted(a for a in attrs if hasattr(mod, a))
    out["compat_names"] = np.array(json.dumps(names))

    # integer bookkeeping on seeded random sizes
    sw = [[cases.digest_list(ref.sampling._sliding_windows(*a))] for a in cases.sliding_window_cases()]
    out["sliding_windows"] = np.array(json.dumps(sw))
    tiles = []
    for h, w, tile, dec in cases.split_tile_cases():
        hook = ref.tilevae.VAEHook(None, tile, is_decoder=dec, fast_decoder=False, fast_encoder=False, color_fix=False)
        with contextlib.redirect_stdout(io.StringIO()):
            rin, rout = hook.split_tiles(h, w)
        crops = []
        for i, o in zip(rin, rout):
            th, tw = i[3] - i[2], i[1] - i[0]
            th, tw = (th * 8, tw * 8) if dec else (th // 8, tw // 8)
            if th > 0 and tw > 0 and h >= 8 and w >= 8:
                idx = torch.arange(th * tw).view(1, 1, th, tw)
                cr = ref.tilevae.crop_valid_region(idx, i, o, dec)
                crops.append([int(cr.shape[2]), int(cr.shape[3]), int(cr[0, 0, 0, 0]) if cr.numel() else -1])
            else:
                crops.append(None)
        tiles.append([cases.digest_list(rin), cases.digest_list(rout), cases.digest_list(crops)])
    out["split_tiles"] = np.array(json.dumps(tiles))
    np.savez_compressed(os.path.join(HERE, "reference_io.npz"), **out)


def gen_engine():
    import pytest
    import make_golden as mg
    import test_dropin_reference_engine_cpu as T
    from sgm.modules.encoders import modules as E
    from SUPIR.models import SUPIR_model as RS
    from weights import make_state_dict
    torch.set_grad_enabled(True)            # batchify_sample manages grad mode itself
    tok_l, tok_g = T.prompt_tokens()
    mp = pytest.MonkeyPatch()
    try:
        with mg.quiet(), mg.cpu_tensor_ctor():
            eng = RS.SUPIRModel(**T.engine_config(T.SAMPLING + "RestoreEDMSampler", False))
            eng.conditioner = mg.build_reference_conditioner(E, tok_l, tok_g, T.ARCH_L, T.ARCH_G, layer_idx=1)
            eng = eng.eval()
            shapes = {k: list(v.shape) for k, v in eng.state_dict().items()}
            sd = make_state_dict(shapes, seed=T.WEIGHT_SEED)
            sigmas = eng.denoiser.sigmas.clone()
            sd["denoiser.sigmas"] = sigmas
            eng.load_state_dict(sd)
            want = T.run_scenarios(eng, mp, untile_reference_hooks=True)
    finally:
        mp.undo()
    out = {k: cases.sample(v).numpy() for k, v in want.items()}
    out.update({k + "_shape": np.array(v.shape) for k, v in want.items()})
    out["shapes"] = np.array(json.dumps(shapes))
    out["sigmas"] = sigmas.numpy()
    np.savez_compressed(os.path.join(HERE, "dropin_engine.npz"), **out)


def gen_options():
    dst = os.path.join(HERE, "options")
    os.makedirs(dst, exist_ok=True)
    for name in sorted(os.listdir(os.path.join(ref_stubs.REFERENCE_ROOT, "options"))):
        if name.endswith(".yaml"):
            shutil.copyfile(os.path.join(ref_stubs.REFERENCE_ROOT, "options", name), os.path.join(dst, name))


if __name__ == "__main__":
    if not ref_stubs.reference_available():
        raise SystemExit(f"no reference checkout at {ref_stubs.REFERENCE_ROOT}: set SUPIR_REFERENCE_ROOT")
    torch.set_grad_enabled(False)
    which = sys.argv[1:] or ["io", "engine", "options"]
    for name in which:
        {"io": gen_io, "engine": gen_engine, "options": gen_options}[name]()

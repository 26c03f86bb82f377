"""Seeded inputs shared by tests/golden/make_reference_io.py (which records the reference's outputs on them) and the tests that
compare this package with those recordings."""
import hashlib
import json
import random

import numpy as np
import torch


def digest(t):
    """sha256 of a tensor's dtype, shape and bytes."""
    t = t.detach().contiguous().cpu()
    h = hashlib.sha256(f"{t.dtype}{tuple(t.shape)}".encode())
    h.update(t.numpy().tobytes())
    return h.hexdigest()


def digest_list(boxes):
    """sha256 of a list of integer boxes (tuples and lists hash alike)."""
    norm = [None if b is None else [int(v) for v in b] for b in boxes]
    return hashlib.sha256(json.dumps(norm).encode()).hexdigest()


def sample(t, n=8192):
    """A fixed, seeded sample of n elements of t (all of them if t is smaller), as float32."""
    flat = t.detach().reshape(-1).float().cpu()
    if flat.numel() <= n:
        return flat
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(flat.numel()))[:n]
    return flat[idx]


def pil2tensor_cases(Image):
    """24 random image sizes x the argument sets test.py / gradio_demo use."""
    rng = random.Random(0)
    for _ in range(24):
        w, h = rng.randint(40, 900), rng.randint(40, 900)
        img = Image.fromarray(np.random.RandomState(w * 1000 + h).randint(0, 255, (h, w, 3), dtype=np.uint8))
        for up, ms, fr in [(1, 1024, None), (2, 1024, None), (4, 64, None), (1, 1024, 512), (3, 256, 512)]:
            yield img, dict(upsacle=up, min_size=ms, fix_resize=fr)


def numpy_helper_inputs():
    rng = np.random.RandomState(0)
    imgs = [rng.randint(0, 256, shape).astype(np.uint8) for shape in ((17, 23), (17, 23, 1), (17, 23, 3), (17, 23, 4))]
    return imgs, rng.randint(0, 256, (9, 11, 3)).astype(np.uint8)


def prepared_conditioner_inputs():
    g = torch.Generator().manual_seed(0)
    c = {"crossattn": torch.randn(1, 77, 32, generator=g), "vector": torch.randn(1, 16, generator=g)}
    uc = {"crossattn": torch.randn(1, 77, 32, generator=g), "vector": torch.randn(1, 16, generator=g)}
    return c, uc, {"control": torch.randn(3, 4, 8, 8, generator=g)}


def sliding_window_cases():
    """(h, w, tile, stride) over the ranges tests/test_properties.py draws from."""
    rng = random.Random(1)
    out = []
    for _ in range(200):
        tile, stride = rng.randint(8, 96), rng.randint(1, 96)
        out.append((tile + rng.randint(0, 700), tile + rng.randint(0, 700), tile, stride))
    return out


def split_tile_cases():
    """(h, w, tile, is_decoder) over the ranges tests/test_properties.py draws from."""
    rng = random.Random(2)
    return [(rng.randint(16, 1200), rng.randint(16, 1200), rng.choice([16, 32, 64, 96, 128, 256, 512]), rng.random() < 0.5)
            for _ in range(150)]

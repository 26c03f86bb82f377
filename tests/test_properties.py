"""Property tests (hypothesis) of the integer bookkeeping on the hot path — window lists, VAE tile boxes, crops, the window
partition over ranks, the network-batch grouping. Bit-exact by nature. The product functions are compared with the oracle's
independent restatement everywhere, and with the reference functions' recorded results on seeded random sizes
(tests/golden/reference_io.npz, tests/golden/make_reference_io.py)."""
import json
import os
import sys

import numpy as np
import torch
from hypothesis import given, settings, strategies as st

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import reference_cases  # noqa: E402

from oracle import sampler as osamp, vae as ovae  # noqa: E402
from supir_b200 import sampling, vae  # noqa: E402

REF = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_io.npz"))


@settings(max_examples=200, deadline=None)
@given(st.integers(8, 96), st.integers(1, 96), st.integers(0, 700), st.integers(0, 700))
def test_sliding_windows_cover_and_match(tile, stride, dh, dw):
    h, w = tile + dh, tile + dw
    got = sampling._sliding_windows(h, w, tile, stride)
    assert [tuple(c) for c in osamp.sliding_windows(h, w, tile, stride)] == got
    # every window is a full tile inside the image, rows/cols are covered, order is row-major
    assert all(he - hi == tile and we - wi == tile and 0 <= hi and he <= h and 0 <= wi and we <= w for hi, he, wi, we in got)
    assert got == sorted(got, key=lambda c: (c[0], c[2]))
    if stride <= tile:       # the reference only guarantees coverage when windows touch or overlap
        rows, cols = set(), set()
        for hi, he, wi, we in got:
            rows.update(range(hi, he)), cols.update(range(wi, we))
        assert rows == set(range(h)) and cols == set(range(w))


@settings(max_examples=150, deadline=None)
@given(st.integers(16, 1200), st.integers(16, 1200), st.sampled_from([16, 32, 64, 96, 128, 256, 512]), st.booleans())
def test_split_tiles_and_crops_match(h, w, tile, dec):
    tin, tout = vae.split_tiles(h, w, tile, dec)
    oin, oout = ovae.split_tiles(h, w, tile, dec)
    assert tin == oin and tout == oout
    # output boxes tile the output canvas exactly once (the paste in tiled_forward relies on it)
    H, W = (h * 8, w * 8) if dec else (h // 8, w // 8)
    area = 0
    for (i, o) in zip(tin, tout):
        x1, x2, y1, y2 = o
        assert 0 <= x1 <= x2 <= W and 0 <= y1 <= y2 <= H
        area += (x2 - x1) * (y2 - y1)
        th, tw = i[3] - i[2], i[1] - i[0]
        th, tw = (th * 8, tw * 8) if dec else (th // 8, tw // 8)
        y0c, y1c, x0c, x1c = vae.crop_margins(th, tw, i, o, dec)
        assert (y0c, y1c, x0c, x1c) == tuple(ovae.crop_margins(th, tw, i, o, dec))
    if not dec and (h % 8 or w % 8):
        return              # the reference floors the latent size; exact tiling is only defined for multiples of 8
    assert area == H * W


def test_sliding_windows_match_the_reference():
    """200 seeded random (h, w, tile, stride) over the ranges above: the window list == the reference's _sliding_windows."""
    want = json.loads(str(REF["sliding_windows"]))
    cases = reference_cases.sliding_window_cases()
    assert len(cases) == len(want)
    for args, (d,) in zip(cases, want):
        assert reference_cases.digest_list(sampling._sliding_windows(*args)) == d, args


def test_split_tiles_and_crops_match_the_reference():
    """150 seeded random (h, w, tile, decoder) over the ranges above: tile boxes == the reference's VAEHook.split_tiles, and the
    crop of every tile (size and first element) == the reference's crop_valid_region on an index image."""
    want = json.loads(str(REF["split_tiles"]))
    cases = reference_cases.split_tile_cases()
    assert len(cases) == len(want)
    for (h, w, tile, dec), (d_in, d_out, d_crop) in zip(cases, want):
        tin, tout = vae.split_tiles(h, w, tile, dec)
        assert reference_cases.digest_list(tin) == d_in and reference_cases.digest_list(tout) == d_out, (h, w, tile, dec)
        crops = []
        for i, o in zip(tin, tout):
            th, tw = i[3] - i[2], i[1] - i[0]
            th, tw = (th * 8, tw * 8) if dec else (th // 8, tw // 8)
            if th > 0 and tw > 0 and h >= 8 and w >= 8:
                y0c, y1c, x0c, x1c = vae.crop_margins(th, tw, i, o, dec)
                crops.append([y1c - y0c, x1c - x0c, y0c * tw + x0c if (y1c - y0c) * (x1c - x0c) > 0 else -1])
            else:
                crops.append(None)
        assert reference_cases.digest_list(crops) == d_crop, (h, w, tile, dec)


@settings(max_examples=300, deadline=None)
@given(st.integers(0, 400), st.integers(1, 16))
def test_shard_windows_is_an_ordered_partition(nw, world):
    spans = [sampling.shard_windows(nw, world, r) for r in range(world)]
    per = spans[0][0]
    assert all(s[0] == per for s in spans) and per * world >= nw
    covered = []
    for r, (_, lo, hi) in enumerate(spans):
        assert lo <= hi <= nw and hi - lo <= per and (lo == min(r * per, nw))
        covered.extend(range(lo, hi))
    assert covered == list(range(nw))           # contiguous blocks in rank order == the reference's window order


@settings(max_examples=300, deadline=None)
@given(st.integers(0, 400), st.integers(1, 64))
def test_balanced_groups(n, cap):
    groups = sampling.balanced_groups(n, cap)
    assert [i for lo, hi in groups for i in range(lo, hi)] == list(range(n))
    sizes = [hi - lo for lo, hi in groups]
    if n:
        assert max(sizes) <= cap and max(sizes) - min(sizes) <= 1 and len(groups) == -(-n // cap)
        assert len(set(sizes)) <= 2             # at most two network batch sizes -> at most two captured graphs


@settings(max_examples=300, deadline=None)
@given(st.integers(0, 600), st.integers(1, 16))
def test_shard_units_balanced_contiguous(n, world):
    spans = [sampling.shard_units(n, world, r) for r in range(world)]
    covered = [u for _, lo, hi in spans for u in range(lo, hi)]
    assert covered == list(range(n))
    sizes = [hi - lo for _, lo, hi in spans]
    assert max(sizes) - min(sizes) <= 1 and all(per == max(sizes) for per, _, _ in spans)


def test_98_units_over_8_ranks():
    """The bench workload's fused-path partition at N = 8: 49 windows x CFG pair = 98 units -> 13, 13, 12 x 6 (no idle rank)."""
    assert [hi - lo for _, lo, hi in (sampling.shard_units(98, 8, r) for r in range(8))] == [13, 13] + [12] * 6
    assert [hi - lo for _, lo, hi in (sampling.shard_units(98, 4, r) for r in range(4))] == [25, 25, 24, 24]


def test_49_windows_over_8_ranks():
    """The generic (foreign-denoiser) path still shards whole windows: seven on ranks 0-6, rank 7 only in the exchange."""
    spans = [sampling.shard_windows(49, 8, r) for r in range(8)]
    assert [hi - lo for _, lo, hi in spans] == [7] * 7 + [0] and spans[0][0] == 7


@settings(max_examples=300, deadline=None)
@given(st.integers(1, 9000), st.integers(8, 2048))
def test_nearest_exact_indices_match_aten(size, tile):
    """The gather indices of the fast tiled-VAE mode's thumbnail (vae.nearest_exact_indices) == the pixels ATen's
    F.interpolate(scale_factor=tile / size, mode='nearest-exact') picks, for every image size / tile size (tilevae.py:859-861)."""
    import torch.nn.functional as F
    if size <= tile:                      # the hook only tiles images larger than one padded tile: scale < 1
        return
    scale = tile / size
    x = torch.arange(size, dtype=torch.float32).view(1, 1, 1, size)
    want = F.interpolate(x, scale_factor=(1.0, scale), mode="nearest-exact")[0, 0, 0].long()
    got = vae.nearest_exact_indices(size, scale)
    assert got.shape == want.shape and torch.equal(got, want), (size, tile)

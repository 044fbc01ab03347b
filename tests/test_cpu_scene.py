"""Host-side parts of whole-scene prediction (nirgan_b200/scene.py): tile grid, row bands, argument checks and the
fp64 blend reference the GPU tests compare against."""
import math

import numpy as np
import pytest
import torch

import nirgan_b200  # noqa: F401
from nirgan_b200 import scene as S
from scene_ref import blend_reference


@pytest.mark.parametrize("H,W,T,ov", [(512, 768, 256, 0),      # aligned, no overlap
                                      (480, 704, 256, 32),     # aligned with overlap: (480 - 256) % 224 == 0
                                      (600, 301, 256, 32),     # unaligned: clamped last tiles
                                      (256, 700, 256, 17),     # H == T: one tile row
                                      (77, 91, 30, 29)])       # stride 1
def test_scene_tiles_grid(H, W, T, ov):
    s = T - ov
    ys, xs = S.scene_grid(H, W, T, ov)
    for n, org in ((H, ys), (W, xs)):
        assert len(org) == math.ceil((n - T) / s) + 1
        assert org[:-1] == [k * s for k in range(len(org) - 1)]
        assert org[-1] == n - T
        assert all(a < b for a, b in zip(org, org[1:]))
    tiles = S.scene_tiles(H, W, T, ov)
    assert tiles == [(y, x) for y in ys for x in xs]
    cover = np.zeros((H, W), dtype=np.int32)
    for y, x in tiles:
        cover[y:y + T, x:x + T] += 1
    assert cover.min() >= 1


@pytest.mark.parametrize("H,W,T,ov", [(255, 300, 256, 0), (300, 255, 256, 0), (300, 300, 256, -1),
                                      (300, 300, 256, 256), (300, 300, 0, 0)])
def test_scene_tiles_rejects_bad_arguments(H, W, T, ov):
    with pytest.raises(ValueError):
        S.scene_tiles(H, W, T, ov)


def _model(**kw):
    from nirgan_b200.config import px2px_config
    from nirgan_b200.model.pix2pix import Px2Px
    c = px2px_config(**kw)
    return c, Px2Px(c).eval()


def test_predict_scene_rejects_tiles_the_generator_refuses():
    _, m = _model()                                   # pad 10: T + 20 must be divisible by 4
    with pytest.raises(ValueError, match="divisible by 4"):
        S.predict_scene(m, torch.zeros(3, 70, 70), tile=66, overlap=0)
    with pytest.raises(ValueError, match="overlap"):
        S.predict_scene(m, torch.zeros(3, 70, 70), tile=64, overlap=64)
    with pytest.raises(ValueError, match="smaller than the tile"):
        S.predict_scene(m, torch.zeros(3, 60, 70), tile=64, overlap=0)
    with pytest.raises(ValueError, match="channels"):
        S.predict_scene(m, torch.zeros(4, 70, 70), tile=64, overlap=0)
    with pytest.raises(ValueError, match="float32 reflectance or uint16"):
        S.predict_scene(m, torch.zeros(3, 70, 70, dtype=torch.float64), tile=64, overlap=0)


def test_predict_scene_embeds_and_satclip_style():
    _, m = _model(inject=True)
    with pytest.raises(ValueError, match="needs embeds"):
        S.predict_scene(m, torch.zeros(3, 70, 70), tile=64, overlap=0)
    with pytest.raises(ValueError, match=r"shape \(4, 256\)"):
        S.predict_scene(m, torch.zeros(3, 70, 70), tile=64, overlap=0, embeds=torch.zeros(3, 256))
    _, plain = _model()
    with pytest.raises(ValueError, match="without SatCLIP"):
        S.predict_scene(plain, torch.zeros(3, 70, 70), tile=64, overlap=0, embeds=torch.zeros(4, 256))
    c, _ = _model(inject=True)
    c.satclip.satclip_style = "concat"
    from nirgan_b200.model.pix2pix import Px2Px
    with pytest.raises(NotImplementedError):
        S.predict_scene(Px2Px(c).eval(), torch.zeros(3, 70, 70), tile=64, overlap=0)


@pytest.mark.parametrize("H", [1, 7, 256, 2048, 8191])
@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_band_split_disjoint_covering_balanced(H, world):
    if world > H:
        with pytest.raises(ValueError):
            S.band_rows(H, 0, world)
        return
    bands = [S.band_rows(H, r, world) for r in range(world)]
    assert bands[0][0] == 0 and bands[-1][1] == H
    assert all(a[1] == b[0] for a, b in zip(bands, bands[1:]))
    sizes = [y1 - y0 for y0, y1 in bands]
    assert max(sizes) - min(sizes) <= 1 and min(sizes) >= 1


@pytest.mark.parametrize("H,T,ov,world", [(2048, 256, 32, 2), (2048, 256, 32, 8), (150, 64, 16, 3), (600, 256, 0, 5),
                                          (256, 256, 32, 4)])
def test_band_tile_set_is_the_intersecting_tiles(H, T, ov, world):
    ys, _ = S.scene_grid(H, T, T, ov)
    for r in range(world):
        y0, y1 = S.band_rows(H, r, world)
        k0, k1 = S.band_tile_rows(ys, T, y0, y1)
        want = {k for k, o in enumerate(ys) if set(range(o, o + T)) & set(range(y0, y1))}
        assert set(range(k0, k1)) == want


def test_assemble_bands_checks_the_tiling():
    parts = [(3, 5, torch.full((1, 2, 4), 1.0)), (0, 3, torch.full((1, 3, 4), 0.0))]
    out = S.assemble_bands(parts)
    assert out.shape == (1, 5, 4) and torch.equal(out[0, :, 0], torch.tensor([0.0, 0, 0, 1, 1]))
    with pytest.raises(ValueError):
        S.assemble_bands([(0, 2, torch.zeros(1, 2, 4)), (3, 5, torch.zeros(1, 2, 4))])


@pytest.mark.parametrize("H,W,T,ov", [(150, 213, 64, 16), (600, 301, 256, 32), (77, 91, 30, 29)])
def test_reference_blend_of_constant_predictions_is_constant(H, W, T, ov):
    ys, xs = S.scene_grid(H, W, T, ov)
    pred = np.full((len(ys) * len(xs), T, T), 0.375)
    out = blend_reference(pred, ys, xs, T, ov, W, 0, H)
    assert out.shape == (H, W)
    assert np.abs(out - 0.375).max() <= 1e-15


def test_reference_blend_without_overlap_on_an_aligned_grid_is_stitching():
    H, W, T = 192, 128, 64
    ys, xs = S.scene_grid(H, W, T, 0)
    pred = np.random.default_rng(0).uniform(-1, 1, (len(ys) * len(xs), T, T))
    out = blend_reference(pred, ys, xs, T, 0, W, 0, H)
    stitched = pred.reshape(len(ys), len(xs), T, T).transpose(0, 2, 1, 3).reshape(H, W)
    assert np.array_equal(out, stitched)

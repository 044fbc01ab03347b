"""Nodata in whole-scene prediction (nirgan_b200/scene.py, `nodata=`): argument checks, and the numpy references of the
nodata mask, the skipped-tile set and the masked blend that the GPU tests compare against."""
import numpy as np
import pytest
import torch

import nirgan_b200  # noqa: F401
from nirgan_b200 import scene as S
from scene_ref import blend_reference


# ---- references --------------------------------------------------------------------------------------------------
def nodata_mask(scene, nodata):
    """(H, W) bool, True where every channel of the (C, H, W) scene equals nodata (NaN matches NaN; float32 scenes
    compare with nodata rounded to fp32)."""
    s = np.asarray(scene)
    if s.dtype == np.uint16:
        return (s.astype(np.int64) == int(nodata)).all(0)
    v = np.float32(nodata)
    return (np.isnan(s) if np.isnan(v) else s == v).all(0)


def tile_counts(valid, origins, T):
    """Valid pixels of each T x T window at origins [(y0, x0), ...] of the (H, W) bool mask `valid`."""
    return np.array([int(valid[y:y + T, x:x + T].sum()) for y, x in origins], dtype=np.int64)


def computed_tiles(valid, H, W, T, overlap):
    """Tile indices (tile-index order) of the tiles with at least one valid pixel: the tiles predict_scene runs."""
    return [t for t, c in enumerate(tile_counts(valid, S.scene_tiles(H, W, T, overlap), T)) if c > 0]


def masked_blend_reference(pred, ys, xs, T, overlap, W, y0, y1, nodata, nodata_out):
    """fp64 blend of the tiles that predict_scene computes, nodata pixels set to nodata_out.  The predictions of
    skipped tiles are replaced by NaN, so a valid pixel that read one would come out NaN."""
    pred = np.array(pred, dtype=np.float64).reshape(len(ys) * len(xs), T, T)
    valid = ~nodata
    for t, (y, x) in enumerate((y, x) for y in ys for x in xs):
        if not valid[y:y + T, x:x + T].any():
            pred[t] = np.nan
    out = blend_reference(pred, ys, xs, T, overlap, W, y0, y1)
    out[nodata[y0:y1]] = nodata_out
    return out


def triangle_pixel_hole(H, W):
    """(H, W) nodata mask: a corner triangle (y / H + x / W < 1.1), one valid pixel inside it at (10, 10), a 5 x 10
    nodata hole in the valid data."""
    yy, xx = np.mgrid[:H, :W]
    nodata = yy * W + xx * H < 1.1 * H * W
    nodata[10, 10] = False
    nodata[120:125, 180:190] = True
    return nodata


# ---- the reference on the masks the GPU tests use ----------------------------------------------------------------
H, W, T, OV = 150, 213, 64, 16           # row origins [0, 48, 86], column origins [0, 48, 96, 144, 149]


def _grid_index(ky, kx):
    return ky * 5 + kx


def test_grid_of_the_reference_scene():
    assert S.scene_grid(H, W, T, OV) == ([0, 48, 86], [0, 48, 96, 144, 149])


def test_whole_nodata_tiles_are_skipped():
    valid = np.ones((H, W), bool)
    valid[:, :100] = False                    # tiles at x0 = 0 (columns 0..63) lie inside; x0 = 48 reaches column 111
    assert computed_tiles(valid, H, W, T, OV) == [t for t in range(15) if t % 5 != 0]
    counts = tile_counts(valid, S.scene_tiles(H, W, T, OV), T)
    assert counts[_grid_index(0, 1)] == 64 * 12 and counts[_grid_index(2, 4)] == 64 * 64


def test_single_valid_pixel_in_a_nodata_region():
    valid = np.zeros((H, W), bool)
    valid[100, 120] = True                    # rows 48..111 and 86..149; columns 96..159 only
    assert computed_tiles(valid, H, W, T, OV) == [_grid_index(1, 2), _grid_index(2, 2)]


def test_nodata_hole_inside_valid_data_skips_nothing():
    valid = np.ones((H, W), bool)
    valid[60:70, 100:110] = False
    assert computed_tiles(valid, H, W, T, OV) == list(range(15))
    assert tile_counts(valid, [(48, 96)], T)[0] == 64 * 64 - 100


def test_triangle_with_a_valid_pixel_and_a_hole():
    # whole tiles (0, 1) and (1, 0) lie in the triangle; (0, 0) is computed for the one valid pixel at (10, 10)
    assert computed_tiles(~triangle_pixel_hole(H, W), H, W, T, OV) == [t for t in range(15) if t not in (1, 5)]
    assert tile_counts(~triangle_pixel_hole(H, W), [(0, 0)], T)[0] == 1


def test_all_nodata_scene_computes_no_tile():
    assert computed_tiles(np.zeros((H, W), bool), H, W, T, OV) == []


def test_nodata_mask_rule():
    s = np.zeros((3, 2, 4), np.float32)
    s[1, 0, 1] = 0.5                          # one channel differs: valid
    s[:, 1, 2] = -0.0                         # -0.0 == 0.0: nodata
    s[:, 1, 3] = np.nan
    m = nodata_mask(s, 0.0)
    assert m.tolist() == [[True, False, True, True], [True, True, True, False]]
    assert nodata_mask(s, float("nan")).tolist() == [[False] * 4, [False, False, False, True]]
    u = np.full((3, 2, 2), 7, np.uint16)
    u[2, 1, 1] = 8
    assert nodata_mask(u, 7).tolist() == [[True, True], [True, False]]


@pytest.mark.parametrize("ov", [16, 0, 40])
def test_masked_reference_reads_no_skipped_tile_at_a_valid_pixel(ov):
    """A tile that covers a valid pixel contains it, so it is never skipped: on a nodata triangle with an isolated
    valid pixel and a hole, the blend with skipped tiles poisoned to NaN is finite at every valid pixel and equals the
    plain blend there."""
    ys, xs = S.scene_grid(H, W, T, ov)
    nodata = triangle_pixel_hole(H, W)
    pred = np.random.default_rng(ov).uniform(-1, 1, (len(ys) * len(xs), T, T))
    out = masked_blend_reference(pred, ys, xs, T, ov, W, 0, H, nodata, -9999.0)
    plain = blend_reference(pred, ys, xs, T, ov, W, 0, H)
    assert np.isfinite(out).all()
    assert np.array_equal(out[~nodata], plain[~nodata])
    assert (out[nodata] == -9999.0).all()
    n_comp = len(computed_tiles(~nodata, H, W, T, ov))
    assert 0 < n_comp < len(ys) * len(xs)


# ---- argument checks ---------------------------------------------------------------------------------------------
def _model(**kw):
    from nirgan_b200.config import px2px_config
    from nirgan_b200.model.pix2pix import Px2Px
    return Px2Px(px2px_config(**kw)).eval()


U16 = torch.zeros(3, 70, 70, dtype=torch.int16).view(torch.uint16)
F32 = torch.zeros(3, 70, 70)


@pytest.mark.parametrize("nodata", [0.5, -1, 65536, float("nan"), float("inf"), "0", True])
def test_uint16_nodata_must_be_an_integer_in_range(nodata):
    with pytest.raises(ValueError, match="nodata"):
        S.predict_scene(_model(), U16, tile=64, overlap=0, nodata=nodata)


@pytest.mark.parametrize("nodata", ["nan", b"0", True, 1j, torch.tensor(0.0), [0.0]])
def test_float32_nodata_must_be_a_real_number(nodata):
    with pytest.raises(ValueError, match="nodata"):
        S.predict_scene(_model(), F32, tile=64, overlap=0, nodata=nodata)


@pytest.mark.parametrize("scene,nodata", [(U16, 0), (U16, 65535), (U16, 0.0), (U16, np.uint16(7)), (F32, 0.0),
                                          (F32, float("nan")), (F32, -9999), (F32, np.float32(-0.0))])
def test_accepted_nodata_reaches_the_device_check(scene, nodata):
    # accepted values pass the argument checks; a CPU model then stops at the device check, before any work
    with pytest.raises(RuntimeError, match="CUDA device"):
        S.predict_scene(_model(), scene, tile=64, overlap=0, nodata=nodata)


def test_nodata_out_must_be_a_number():
    with pytest.raises(ValueError, match="nodata_out"):
        S.predict_scene(_model(), U16, tile=64, overlap=0, nodata=0, nodata_out="nan")


@pytest.mark.parametrize("nodata", [None, 0])
def test_existing_checks_hold_with_and_without_nodata(nodata):
    m = _model()
    with pytest.raises(ValueError, match="divisible by 4"):
        S.predict_scene(m, U16, tile=66, overlap=0, nodata=nodata)
    with pytest.raises(ValueError, match="overlap"):
        S.predict_scene(m, U16, tile=64, overlap=64, nodata=nodata)
    with pytest.raises(ValueError, match="smaller than the tile"):
        S.predict_scene(m, torch.zeros(3, 60, 70), tile=64, overlap=0, nodata=nodata)
    with pytest.raises(ValueError, match="channels"):
        S.predict_scene(m, torch.zeros(4, 70, 70), tile=64, overlap=0, nodata=nodata)
    with pytest.raises(ValueError, match="float32 reflectance or uint16"):
        S.predict_scene(m, torch.zeros(3, 70, 70, dtype=torch.float64), tile=64, overlap=0, nodata=nodata)
    with pytest.raises(ValueError, match="needs embeds"):
        S.predict_scene(_model(inject=True), U16, tile=64, overlap=0, nodata=nodata)
